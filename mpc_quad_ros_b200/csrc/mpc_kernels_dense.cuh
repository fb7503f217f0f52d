// mpc_kernels_dense.cuh — K2b: condensed (dense) box-QP solver, one CTA per OCP, for the OCPs whose warm-started
// active-set rounds did not settle in the screening kernel (qmpc_ipm_kernel with a hard list) and for cold starts.
//
// Why: a Riccati sweep is 20 strictly sequential stages of warp-serial work; the ~5 % of OCPs that need the
// interior-point method kept one warp busy for 1.3-2.7 ms while the rest of the GPU idled (profiles/r01_timeline.txt).
// Eliminating the states gives  min 1/2 du' H du + f' du,  lb <= ubar + du <= ub  with H = Rbar + sum_k G_k' Q_k G_k
// (G_k = impulse responses), E = 4N <= 88 unknowns.  Everything is then wide: condensing is 4x4-tile rank-13 updates
// held in registers (one thread per tile of the lower triangle), every factorisation is a blocked Cholesky over the
// same tiles (2 barriers per block column), gradients/multipliers are dense mat-vecs; only the two triangular solves
// per right-hand side stay serial (one warp, shuffles).  Same algorithm as the Riccati path: Mehrotra IPM from the
// box centre with gradient-scaled multipliers, hand-over to exact primal-dual active-set rounds, full step.
#pragma once
#include "mpc_kernels.cuh"

// build-time variants (A/B): see the functions they select
#ifndef QMPC_DENSE_FACTOR
#define QMPC_DENSE_FACTOR 1         // 2: tile per thread, one barrier per block column (factor_rl1); 1: column per warp, flags (factor_cols); 0: two barriers (factor)
#endif
#ifndef QMPC_DENSE_SCALED_SOLVE
#define QMPC_DENSE_SCALED_SOLVE 1   // triangular sweeps on tiles pre-scaled by their column's diagonal inverse (scale_for_solves); 0: plain sweeps
#endif
#ifndef QMPC_DENSE_UNROLL
#define QMPC_DENSE_UNROLL 2         // unroll factor of the H x and triangular-sweep loops (2: the next step's tile loads overlap the chain)
#endif
#ifndef QMPC_DENSE_GPLANES
#define QMPC_DENSE_GPLANES 1        // condensing: impulse-response rows stored as two planes (see gcol)
#endif
#ifndef QMPC_DENSE_MATVEC2
#define QMPC_DENSE_MATVEC2 0        // 1: two threads per row of H x (measured slower under load: -2.7 %, profiles/r02_policy_ab.txt)
#endif

namespace qmpc {

constexpr int DN_THREADS = 256;
constexpr int DN_UNROLL = QMPC_DENSE_UNROLL;
constexpr int DN_MAX_N = 21;        // N(N+1)/2 tiles + N right-hand-side threads <= 256
constexpr int TS = 18;              // reals per 4x4 tile in shared memory: 144 B stride spreads consecutive tiles over the banks

template <typename real>
struct DenseArgs {
    IpmArgs<real> b;
    const int* hard_list;           // OCP indices to solve, or null = all of 0..B-1
    const int* hard_count;          // device counter written by the screening kernel (read here, no host sync)
    int* next_item;                 // work queue: CTAs take their first item by index and every further one from this counter
                                    // (zeroed before the launch; IPM and round counts vary 6x between OCPs), or null = strided
};

// shared-memory carve-up (reals).  Condensing works in a region that OVERLAYS Ht/Lt (written when it ends):
//   tiles[N][13][16]          all stage tiles of the OCP, fetched with one TMA bulk copy (cp.async.bulk + mbarrier)
//   Gc[2][DN_CH][13][GS]      sqrt(Q)-scaled impulse-response columns of DN_CH stages, double-buffered
//   evc[2][DN_CH][16]         sqrt(Q)-scaled free response + (iterate - reference) of those stages
struct DenseLayout {
    int E, T, GS, Ht, Lt, tiles, Gc, evc, sq, sml, cbar, dxs, vec, total;
};
constexpr int DN_NVEC = 18;
constexpr int DN_CH = 3;            // stages per condensing chunk (one CTA barrier per chunk)
__host__ __device__ inline DenseLayout dense_layout(int N)
{
    DenseLayout L;
    L.E = 4 * N; L.T = N * (N + 1) / 2; L.GS = L.E + 4;
    L.Ht = 0; L.Lt = L.T * TS;
    L.tiles = 0; L.Gc = N * WT; L.evc = L.Gc + 2 * DN_CH * 13 * L.GS;
    const int cond = L.evc + 2 * DN_CH * 16, fact = 2 * L.T * TS;
    L.sq = cond > fact ? cond : fact;
    L.sml = L.sq + 32;                   // small: wv(16) xp(16) reduction scratch(16) control words(8) mbarrier(8)
    L.cbar = L.sml + 64;                 // one completion flag (mbarrier) per block column of the factorisation
    L.dxs = L.cbar + DN_MAX_N + 3;
    L.vec = (L.dxs + 13 * (N + 1) + 1) & ~1;
    L.total = L.vec + DN_NVEC * L.E;
    return L;
}

__device__ __forceinline__ int tri(int i, int j) { return i * (i + 1) / 2 + j; }   // tile (i, j), j <= i

// inverse of a 4x4 Cholesky factor (lower triangular, row-major packed): triangular solves become short products
template <typename real>
struct Inv4 {
    real n00, n10, n11, n20, n21, n22, n30, n31, n32, n33;
    __device__ __forceinline__ void from(const Chol4<real>& L)
    {
        n00 = L.i0; n11 = L.i1; n22 = L.i2; n33 = L.i3;
        n10 = -L.l10 * n00 * n11;
        n21 = -L.l21 * n11 * n22;
        n32 = -L.l32 * n22 * n33;
        n20 = -(L.l20 * n00 + L.l21 * n10) * n22;
        n31 = -(L.l31 * n11 + L.l32 * n21) * n33;
        n30 = -(L.l30 * n00 + L.l31 * n10 + L.l32 * n20) * n33;
    }
    __device__ __forceinline__ void store(real* p) const
    {
        p[0] = n00; p[1] = n10; p[2] = n11; p[3] = n20; p[4] = n21; p[5] = n22; p[6] = n30; p[7] = n31; p[8] = n32; p[9] = n33;
    }
    __device__ __forceinline__ void load(const real* p)
    {
        ld2(p, n00, n10); ld2(p + 2, n11, n20); ld2(p + 4, n21, n22); ld2(p + 6, n30, n31); ld2(p + 8, n32, n33);
    }
    __device__ __forceinline__ void mul(const real* v, real* z) const      // z = Lam^-1 v
    {
        z[0] = n00 * v[0];
        z[1] = n10 * v[0] + n11 * v[1];
        z[2] = (n20 * v[0] + n21 * v[1]) + n22 * v[2];
        z[3] = (n30 * v[0] + n31 * v[1]) + (n32 * v[2] + n33 * v[3]);
    }
    __device__ __forceinline__ void mulT(const real* v, real* z) const     // z = Lam^-T v
    {
        z[0] = (n00 * v[0] + n10 * v[1]) + (n20 * v[2] + n30 * v[3]);
        z[1] = (n11 * v[1] + n21 * v[2]) + n31 * v[3];
        z[2] = n22 * v[2] + n32 * v[3];
        z[3] = n33 * v[3];
    }
};

// The column-per-warp factorisation of DenseCtx::factor_cols (described there), as a free function that is NOT inlined.
template <typename real>
#ifdef QMPC_FCOLS_INLINE
__device__ __forceinline__
#else
__device__ __noinline__
#endif
void factor_cols_fn(const int oHt, const int oLt, const int oRt, const int oFx, const int oDR, const int oCbar,
                    const unsigned fgen, const int N, const int tid, const bool fixed)
{
    // the arrays arrive as offsets into the CTA's dynamic shared memory and are rebuilt from the shared symbol here:
    // pointer arguments of a non-inlined function are generic, and every access would be a generic LD / ST
    QMPC_DYN_SMEM(smem_raw);
    real* const sm = reinterpret_cast<real*>(smem_raw);
    const real* const Ht = sm + oHt;
    real* const Lt = sm + oLt;
    real* const rt = sm + oRt;
    const real* const fx = sm + oFx;
    const real* const dR = sm + oDR;
    unsigned long long* const cbar = reinterpret_cast<unsigned long long*>(sm + oCbar);
    const int warp = tid >> 5, lane = tid & 31;
    for (int j = warp; j < N; j += DN_THREADS / 32) {
        const int rows = N - j;
        const bool tile = lane > 0 && lane < rows, rhs = lane == rows;
        const int i = tile ? j + lane : j;
        // dg: the diagonal tile (j, j), carried REDUNDANTLY by every lane (lower triangle); acc: this lane's own tile
        real acc[16], dg[16];
        real kj[4] = {1, 1, 1, 1};
        {
            const real* p = Ht + tri(j, j) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, dg[t], dg[t + 1]);
            if (fixed) {
#pragma unroll
                for (int q = 0; q < 4; ++q) kj[q] = fx[4 * j + q] != real(0) ? real(0) : real(1);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 4; ++r) dg[q * 4 + r] *= kj[q] * kj[r];
#pragma unroll
                for (int q = 0; q < 4; ++q) if (kj[q] == real(0)) dg[q * 5] = real(1);
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) dg[q * 5] += dR[4 * j + q];
            }
        }
#pragma unroll
        for (int t = 0; t < 16; ++t) acc[t] = 0;
        if (tile) {
            const real* p = Ht + tri(i, j) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, acc[t], acc[t + 1]);
            if (fixed) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const real ki = fx[4 * i + q] != real(0) ? real(0) : real(1);
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[q * 4 + r] *= ki * kj[r];
                }
            }
        } else if (rhs) {
            ld2(rt + 4 * j, acc[0], acc[1]); ld2(rt + 4 * j + 2, acc[2], acc[3]);
        }
        for (int k = 0; k < j - 1; ++k) {       // look-ahead: columns finished long ago
            flag_wait(cbar + k, fgen);
            real lj[16];
            const real* pj = Lt + tri(j, k) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(pj + t, lj[t], lj[t + 1]);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int r = 0; r <= q; ++r) {
                    real s = dg[q * 4 + r];
#pragma unroll
                    for (int c = 0; c < 4; ++c) s = fma(-lj[q * 4 + c], lj[r * 4 + c], s);
                    dg[q * 4 + r] = s;
                }
            // row q of this lane's left factor: tile (i, k), or the forward-substituted right-hand side of block k
            const real* pi = rhs ? rt + 4 * k : Lt + tri(i, k) * TS;
            const int nq = rhs ? 1 : (tile ? 4 : 0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (q < nq) {
                    real l0, l1, l2, l3;
                    ld2(pi + q * 4, l0, l1); ld2(pi + q * 4 + 2, l2, l3);
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        real s = acc[q * 4 + r];
                        s = fma(-l0, lj[r * 4], s); s = fma(-l1, lj[r * 4 + 1], s);
                        s = fma(-l2, lj[r * 4 + 2], s); s = fma(-l3, lj[r * 4 + 3], s);
                        acc[q * 4 + r] = s;
                    }
                }
            }
        }
        // The column that has just finished (k = j - 1) is the serial chain of the whole factorisation: its product, the
        // 4x4 Cholesky of the diagonal tile and the substitution of this lane's rows form ONE basic block (no branch:
        // idle lanes compute on valid dummy addresses, the reciprocal square roots are branch-free), so the scheduler
        // moves the 64 FMAs of the lane's own tile into the latency of the Cholesky's dependent chain.
        if (j > 0) {
            const int k = j - 1;
            flag_wait(cbar + k, fgen);
            real lj[16];
            const real* pj = Lt + tri(j, k) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(pj + t, lj[t], lj[t + 1]);
            const real* pi = rhs ? rt + 4 * k : Lt + tri(i, k) * TS;      // i == j for lanes without a tile: a valid address
            const int qs = rhs ? 0 : 4;             // the right-hand-side lane has one row: it reads it four times (rows 1..3 unused)
            real li[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) { ld2(pi + q * qs, li[q * 4], li[q * 4 + 1]); ld2(pi + q * qs + 2, li[q * 4 + 2], li[q * 4 + 3]); }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int r = 0; r <= q; ++r) {
                    real s = dg[q * 4 + r];
#pragma unroll
                    for (int c = 0; c < 4; ++c) s = fma(-lj[q * 4 + c], lj[r * 4 + c], s);
                    dg[q * 4 + r] = s;
                }
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int r = 0; r < 4; ++r) {
                    real s = acc[q * 4 + r];
#pragma unroll
                    for (int c = 0; c < 4; ++c) s = fma(-li[q * 4 + c], lj[r * 4 + c], s);
                    acc[q * 4 + r] = s;
                }
        }
        // every lane factors the diagonal tile itself: no broadcast, no warp barrier
        Chol4<real> L;
        L.template factor<real, true>(dg);
        real z[16];
#pragma unroll
        for (int q = 0; q < 4; ++q) L.fsolve(acc + q * 4, z + q * 4);
        if (tile) {
            real* o = Lt + tri(i, j) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) st2(o + t, z[t], z[t + 1]);
        } else if (rhs) {
            st2(rt + 4 * j, z[0], z[1]); st2(rt + 4 * j + 2, z[2], z[3]);
        }
        flag_arrive(cbar + j);
        if (lane == 0) {            // the inverse of the diagonal factor is only read by solve(), after the closing barrier
            Inv4<real> Ni;
            Ni.from(L);
            Ni.store(Lt + tri(j, j) * TS);
        }
    }
    __syncthreads();
}


template <typename real>
struct DenseCtx {
    const IpmArgs<real>& a;
    int tid, lane, N, E, T, GS, ti, tj;
    int fi, fj;                     // factor_rl1's own thread -> tile map (fj < 0: no work)
    real *Ht, *Lt;
    real *f, *ubar, *ucur, *tl, *tu, *ll, *lu, *cl, *cu, *ua, *usol, *rt, *dR, *tv, *itl, *itu, *ill, *ilu, *fx, *fv;
    real* smbase;                   // start of the CTA's dynamic shared memory
    unsigned long long* cbar;       // completion flag of every block column (factor_cols)
    unsigned fgen;                  // factorisations done so far by this CTA = generation of the flags

    // tv = H x  (H symmetric, stored as 4x4 tiles of the lower triangle).  Two threads per row - the even and the odd block
    // columns - combined with one shuffle; whole warps take part (rows past the end are computed redundantly, not stored).
    __device__ __forceinline__ void matvec(const real* x)
    {
#if QMPC_DENSE_MATVEC2
        const int nthr = (2 * E + 31) & ~31;
        if (tid < nthr) {
            const int row = (tid >> 1) < E ? (tid >> 1) : E - 1, half = tid & 1;
            const int I = row >> 2, ar = row & 3;
            real s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll 2
            for (int J = half; J <= I; J += 2) {
                const real* p = Ht + tri(I, J) * TS + ar * 4;
                real h0, h1, h2, h3, x0, x1, x2, x3;
                ld2(p, h0, h1); ld2(p + 2, h2, h3);
                ld2(x + 4 * J, x0, x1); ld2(x + 4 * J + 2, x2, x3);
                s0 = fma(h0, x0, s0); s1 = fma(h1, x1, s1); s2 = fma(h2, x2, s2); s3 = fma(h3, x3, s3);
            }
#pragma unroll 2
            for (int J = I + 1 + ((I + 1 + half) & 1); J < N; J += 2) {       // first J > I with J == half (mod 2)
                const real* p = Ht + tri(J, I) * TS + ar;
                real x0, x1, x2, x3;
                ld2(x + 4 * J, x0, x1); ld2(x + 4 * J + 2, x2, x3);
                s0 = fma(p[0], x0, s0); s1 = fma(p[4], x1, s1); s2 = fma(p[8], x2, s2); s3 = fma(p[12], x3, s3);
            }
            real s = (s0 + s1) + (s2 + s3);
            s += __shfl_xor_sync(FULL, s, 1);
            if (half == 0 && (tid >> 1) < E) tv[row] = s;
        }
#else
        if (tid < E) {
            const int I = tid >> 2, ar = tid & 3;
            real s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll DN_UNROLL
            for (int J = 0; J <= I; ++J) {
                const real* p = Ht + tri(I, J) * TS + ar * 4;
                real h0, h1, h2, h3, x0, x1, x2, x3;
                ld2(p, h0, h1); ld2(p + 2, h2, h3);
                ld2(x + 4 * J, x0, x1); ld2(x + 4 * J + 2, x2, x3);
                s0 = fma(h0, x0, s0); s1 = fma(h1, x1, s1); s2 = fma(h2, x2, s2); s3 = fma(h3, x3, s3);
            }
#pragma unroll DN_UNROLL
            for (int J = I + 1; J < N; ++J) {
                const real* p = Ht + tri(J, I) * TS + ar;
                real x0, x1, x2, x3;
                ld2(x + 4 * J, x0, x1); ld2(x + 4 * J + 2, x2, x3);
                s0 = fma(p[0], x0, s0); s1 = fma(p[4], x1, s1); s2 = fma(p[8], x2, s2); s3 = fma(p[12], x3, s3);
            }
            tv[tid] = (s0 + s1) + (s2 + s3);
        }
#endif
    }

    // NOT inlined on purpose: inside the kernel the register allocator has the solver's ~25 vector pointers live across the
    // call and schedules this loop 60 % slower than the same code compiled on its own (38.7 k against 23.6 k cycles per
    // factorisation, scripts/ubench/factor.cu)
    __device__ __forceinline__ void factor_cols(const bool fixed)
    {
        factor_cols_fn<real>(int(Ht - smbase), int(Lt - smbase), int(rt - smbase), int(fx - smbase), int(dR - smbase),
                             int(reinterpret_cast<real*>(cbar) - smbase), fgen, N, tid, fixed);
        ++fgen;
    }

    // Right-looking, one thread per 4x4 tile, ONE CTA barrier per block column (QMPC_DENSE_FACTOR 2).  A warp-level
    // fp64 instruction occupies the SMSP's fp64 pipe for two cycles however few lanes are active, so the mapping packs
    // the active lanes: tiles are numbered column-major (see the kernel prologue).  Every thread of
    // block column c (its tiles and the right-hand-side thread of block c) also carries the diagonal tile (c, c): the
    // update with column K subtracts L(c,K) L(c,K)' from it - the thread has loaded L(c,K) anyway - so when column c
    // becomes current each of its threads factors the diagonal tile itself and substitutes its own rows at once.  The
    // separate panel phase of the variant below (a second barrier per block column, one thread factoring while 255 wait)
    // is gone; the price is 40 more FMAs per tile update.
    __device__ __forceinline__ void factor_rl1(const bool fixed)
    {
        // thread -> (row fi, column fj) of the factorisation, COLUMN-major: the N - c tiles of block column c and its
        // right-hand-side thread (fi == N) are consecutive threads, so the threads that factor the current column sit
        // in one or two warps and the warps whose columns are finished drop out of the updates entirely
        const bool work = fj >= 0, rhs = work && fi == N, tile = work && !rhs;
        const int col = work ? fj : 0, ti = tile ? fi : 0;
        const bool below = tile && fi > fj;
        const int tix = tri(ti, col);       // tile index in Ht / Lt
        real acc[16], dg[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) { acc[t] = 0; dg[t] = 0; }
        if (work) {
            real kj[4] = {1, 1, 1, 1};
            const real* p = Ht + tri(col, col) * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, dg[t], dg[t + 1]);
            if (fixed) {
#pragma unroll
                for (int q = 0; q < 4; ++q) kj[q] = fx[4 * col + q] != real(0) ? real(0) : real(1);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 4; ++r) dg[q * 4 + r] *= kj[q] * kj[r];
#pragma unroll
                for (int q = 0; q < 4; ++q) if (kj[q] == real(0)) dg[q * 5] = real(1);
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) dg[q * 5] += dR[4 * col + q];
            }
            if (below) {
                const real* pa = Ht + tix * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(pa + t, acc[t], acc[t + 1]);
                if (fixed) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const real ki = fx[4 * ti + q] != real(0) ? real(0) : real(1);
#pragma unroll
                        for (int r = 0; r < 4; ++r) acc[q * 4 + r] *= ki * kj[r];
                    }
                }
            } else if (rhs) {
                ld2(rt + 4 * col, acc[0], acc[1]); ld2(rt + 4 * col + 2, acc[2], acc[3]);
            }
        }
        for (int K = 0; K < N; ++K) {
            const bool current = work && col == K;
            Chol4<real> L;
            if (current) {
                L.factor(dg);
                L.pin();
                if (below) {
                    real* o = Lt + tix * TS;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        real z[4];
                        L.fsolve(acc + q * 4, z);
                        st2(o + q * 4, z[0], z[1]); st2(o + q * 4 + 2, z[2], z[3]);
                    }
                } else if (rhs) {
                    real y[4];
                    L.fsolve(acc, y);
                    st2(rt + 4 * K, y[0], y[1]); st2(rt + 4 * K + 2, y[2], y[3]);
                }
            }
            __syncthreads();
            if (current && tile && !below) {    // the diagonal thread: the inverse is only read by solve(), after the last barrier
                Inv4<real> Ni;
                Ni.from(L);
                Ni.store(Lt + tix * TS);
            }
            if (work && col > K) {
                real lj[16];
                const real* pj = Lt + tri(col, K) * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(pj + t, lj[t], lj[t + 1]);
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r <= q; ++r) {
                        real s = dg[q * 4 + r];
#pragma unroll
                        for (int c = 0; c < 4; ++c) s = fma(-lj[q * 4 + c], lj[r * 4 + c], s);
                        dg[q * 4 + r] = s;
                    }
                const real* pi = rhs ? rt + 4 * K : Lt + tri(ti, K) * TS;
                const int nq = rhs ? 1 : (below ? 4 : 0);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (q < nq) {
                        real l0, l1, l2, l3;
                        ld2(pi + q * 4, l0, l1); ld2(pi + q * 4 + 2, l2, l3);
#pragma unroll
                        for (int r = 0; r < 4; ++r) {
                            real s = acc[q * 4 + r];
                            s = fma(-l0, lj[r * 4], s); s = fma(-l1, lj[r * 4 + 1], s);
                            s = fma(-l2, lj[r * 4 + 2], s); s = fma(-l3, lj[r * 4 + 3], s);
                            acc[q * 4 + r] = s;
                        }
                    }
                }
            }
        }
        __syncthreads();        // the last diagonal inverse is visible to solve()
    }

    // Right-looking variant (QMPC_DENSE_FACTOR 0), same result: one thread per 4x4 tile; the current panel goes through
    // shared memory and the next diagonal block is factored while the other tiles take their update (two CTA barriers
    // per block column).  Threads T..T+N-1 carry the right-hand side.
    __device__ __forceinline__ void factor(const bool fixed)
    {
        real acc[16];
        real r4[4] = {0, 0, 0, 0};
        const bool tile = tid < T, rhs = tid >= T && tid < T + N;
        const int J = tid - T;
        if (tile) {
            const real* p = Ht + tid * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, acc[t], acc[t + 1]);
            if (fixed) {
                real ki[4], kj[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    ki[q] = fx[4 * ti + q] != real(0) ? real(0) : real(1);
                    kj[q] = fx[4 * tj + q] != real(0) ? real(0) : real(1);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[q * 4 + r] *= ki[q] * kj[r];
                if (ti == tj) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) if (ki[q] == real(0)) acc[q * 5] = real(1);
                }
            } else if (ti == tj) {
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[q * 5] += dR[4 * ti + q];
            }
        } else if (rhs) {
            ld2(rt + 4 * J, r4[0], r4[1]); ld2(rt + 4 * J + 2, r4[2], r4[3]);
        }
        if (tid == 0) {
            Chol4<real> L;
#if QMPC_RSQRT_NOBRANCH
            L.template factor<real, true>(acc);
#else
            L.factor(acc);
#endif
            Inv4<real> Ni;
            Ni.from(L);
            Ni.store(Lt);
        }
        __syncthreads();
        for (int K = 0; K < N; ++K) {
            if (tile && tj == K && ti > K) {
                Inv4<real> Ni;
                Ni.load(Lt + tri(K, K) * TS);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    real z[4];
                    Ni.mul(acc + q * 4, z);
#pragma unroll
                    for (int r = 0; r < 4; ++r) acc[q * 4 + r] = z[r];
                }
                real* o = Lt + tid * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) st2(o + t, acc[t], acc[t + 1]);
            } else if (rhs && J == K) {
                Inv4<real> Ni;
                Ni.load(Lt + tri(K, K) * TS);
                real y[4];
                Ni.mul(r4, y);
                st2(rt + 4 * K, y[0], y[1]); st2(rt + 4 * K + 2, y[2], y[3]);
            }
            __syncthreads();
            if (tile && tj > K) {
                real li[16], lj[16];
                const real* pi = Lt + tri(ti, K) * TS;
                const real* pj = Lt + tri(tj, K) * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) { ld2(pi + t, li[t], li[t + 1]); ld2(pj + t, lj[t], lj[t + 1]); }
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        real s = acc[q * 4 + r];
#pragma unroll
                        for (int c = 0; c < 4; ++c) s = fma(-li[q * 4 + c], lj[r * 4 + c], s);
                        acc[q * 4 + r] = s;
                    }
                if (ti == K + 1 && tj == K + 1) {
                    Chol4<real> L;
        #if QMPC_RSQRT_NOBRANCH
            L.template factor<real, true>(acc);
#else
            L.factor(acc);
#endif
                    Inv4<real> Ni;
                    Ni.from(L);
                    Ni.store(Lt + tid * TS);
                }
            } else if (rhs && J > K) {
                real lj[16], y[4];
                const real* pj = Lt + tri(J, K) * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(pj + t, lj[t], lj[t + 1]);
                ld2(rt + 4 * K, y[0], y[1]); ld2(rt + 4 * K + 2, y[2], y[3]);
#pragma unroll
                for (int q = 0; q < 4; ++q) r4[q] -= (lj[q * 4] * y[0] + lj[q * 4 + 1] * y[1]) + (lj[q * 4 + 2] * y[2] + lj[q * 4 + 3] * y[3]);
            }
            __syncthreads();
        }
    }

#if QMPC_DENSE_SCALED_SOLVE
    // After the factorisation (all threads): every off-diagonal tile L(i,j) becomes V(i,j) = L(i,j) Lam_j^-1, scaled by the
    // inverse of its COLUMN's diagonal factor.  Both triangular sweeps then run on the pre-scaled residuals:
    //   forward   s_J = r_J - sum_{I<J} V(J,I) s_I,            y_J = Lam_J^-1 s_J   once, at the end
    //   backward  x_K = Lam_K^-T y_K - sum_{I>K} V(I,K)' x_I   (the first term once, at the start)
    // so a step of the serial chain is one shuffle of four values and one 4x4 product; the product with the diagonal
    // inverse (16 more dependent fp64 operations per step, issued by one warp) is off the chain.  8.2 k -> see DESIGN.
    __device__ __forceinline__ void scale_for_solves()
    {
        if (tid < T && ti > tj) {
            Inv4<real> Ni;
            Ni.load(Lt + tri(tj, tj) * TS);
            real* p = Lt + tid * TS;
            real l[16], z[16];
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, l[t], l[t + 1]);
#pragma unroll
            for (int q = 0; q < 4; ++q) Ni.mulT(l + q * 4, z + q * 4);      // row q of L Lam^-1
#pragma unroll
            for (int t = 0; t < 16; t += 2) st2(p + t, z[t], z[t + 1]);
        }
        __syncthreads();
    }

    // warp 0, lane I < N owns block row I: dst = K^-1 rhs with the scaled factor in Lt; fwd_done: rhs already holds Lam^-1 rhs
    __device__ __forceinline__ void solve(const real* rhs, real* dst, const bool fwd_done)
    {
        real r4[4] = {0, 0, 0, 0};
        const int me = lane < N ? lane : N - 1;         // lanes past the last block row compute on row N-1 and store nothing
        ld2(rhs + 4 * me, r4[0], r4[1]); ld2(rhs + 4 * me + 2, r4[2], r4[3]);
        Inv4<real> Nme;
        Nme.load(Lt + tri(me, me) * TS);
        if (!fwd_done) {
#pragma unroll DN_UNROLL
            for (int K = 0; K < N - 1; ++K) {
                const real* p = Lt + tri(me > K ? me : K + 1, K) * TS;       // a valid tile for every lane
                real l[16], sk[4];
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(p + t, l[t], l[t + 1]);
#pragma unroll
                for (int q = 0; q < 4; ++q) sk[q] = __shfl_sync(FULL, r4[q], K);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const real upd = r4[q] - ((l[q * 4] * sk[0] + l[q * 4 + 1] * sk[1]) + (l[q * 4 + 2] * sk[2] + l[q * 4 + 3] * sk[3]));
                    r4[q] = me > K ? upd : r4[q];
                }
            }
            real y[4];
            Nme.mul(r4, y);
#pragma unroll
            for (int q = 0; q < 4; ++q) r4[q] = y[q];
        }
        {
            real x[4];
            Nme.mulT(r4, x);
#pragma unroll
            for (int q = 0; q < 4; ++q) r4[q] = x[q];
        }
#pragma unroll DN_UNROLL
        for (int K = N - 1; K > 0; --K) {
            const real* p = Lt + tri(K, me < K ? me : K - 1) * TS;
            real l[16], xk[4];
#pragma unroll
            for (int t = 0; t < 16; t += 2) ld2(p + t, l[t], l[t + 1]);
#pragma unroll
            for (int q = 0; q < 4; ++q) xk[q] = __shfl_sync(FULL, r4[q], K);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const real upd = r4[c] - ((l[c] * xk[0] + l[4 + c] * xk[1]) + (l[8 + c] * xk[2] + l[12 + c] * xk[3]));
                r4[c] = me < K ? upd : r4[c];
            }
        }
        if (lane < N) { st2(dst + 4 * lane, r4[0], r4[1]); st2(dst + 4 * lane + 2, r4[2], r4[3]); }
        __syncwarp();
    }
#else
    __device__ __forceinline__ void scale_for_solves() {}
    // warp 0, lane I < N owns block row I: dst = K^-1 rhs with the factor in Lt; fwd_done: rhs already holds Lam^-1 rhs
    __device__ __forceinline__ void solve(const real* rhs, real* dst, const bool fwd_done)
    {
        real r4[4] = {0, 0, 0, 0};
        const bool row = lane < N;
        if (row) { ld2(rhs + 4 * lane, r4[0], r4[1]); ld2(rhs + 4 * lane + 2, r4[2], r4[3]); }
        if (!fwd_done) {
            for (int K = 0; K < N; ++K) {
                real l[16];
                if (row && lane > K) {
                    const real* p = Lt + tri(lane, K) * TS;
#pragma unroll
                    for (int t = 0; t < 16; t += 2) ld2(p + t, l[t], l[t + 1]);
                } else {
#pragma unroll
                    for (int t = 0; t < 16; ++t) l[t] = 0;
                }
                Inv4<real> Ni;
                Ni.load(Lt + tri(K, K) * TS);
                real rk[4], y[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) rk[q] = __shfl_sync(FULL, r4[q], K);
                Ni.mul(rk, y);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const real upd = r4[q] - ((l[q * 4] * y[0] + l[q * 4 + 1] * y[1]) + (l[q * 4 + 2] * y[2] + l[q * 4 + 3] * y[3]));
                    r4[q] = lane == K ? y[q] : upd;
                }
            }
        }
        for (int K = N - 1; K >= 0; --K) {
            real l[16];
            if (lane < K) {
                const real* p = Lt + tri(K, lane) * TS;
#pragma unroll
                for (int t = 0; t < 16; t += 2) ld2(p + t, l[t], l[t + 1]);
            } else {
#pragma unroll
                for (int t = 0; t < 16; ++t) l[t] = 0;
            }
            Inv4<real> Ni;
            Ni.load(Lt + tri(K, K) * TS);
            real rk[4], x[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) rk[q] = __shfl_sync(FULL, r4[q], K);
            Ni.mulT(rk, x);
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const real upd = r4[c] - ((l[c] * x[0] + l[4 + c] * x[1]) + (l[8 + c] * x[2] + l[12 + c] * x[3]));
                r4[c] = lane == K ? x[c] : upd;
            }
        }
        if (row) { st2(dst + 4 * lane, r4[0], r4[1]); st2(dst + 4 * lane + 2, r4[2], r4[3]); }
        __syncwarp();
    }
#endif
};

#ifdef QMPC_DENSE_PROF
#define DPROF_DECL long long pf_t0 = clock64(), pf_last = pf_t0, pf_acc[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}; int pf_n[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
#define DPROF(slot) { const long long pf_now = clock64(); pf_acc[slot] += pf_now - pf_last; ++pf_n[slot]; pf_last = pf_now; }
#else
#define DPROF_DECL
#define DPROF(slot)
#endif

// element loop of warp 0: e = lane, lane + 32, lane + 64 (E <= 96), unrolled so the three elements overlap
#define DN_FOR_E(e) _Pragma("unroll") for (int e##_m = 0; e##_m < 3; ++e##_m) for (int e = lane + 32 * e##_m; e < E; e = E)

#ifndef QMPC_DENSE_MIN_CTAS
#define QMPC_DENSE_MIN_CTAS 2       // register budget: 2 -> 128 registers per thread
#endif

template <typename real>
__global__ void __launch_bounds__(DN_THREADS, QMPC_DENSE_MIN_CTAS) qmpc_dense_kernel(DenseArgs<real> da)
{
    QMPC_DYN_SMEM(smem_raw);
    const IpmArgs<real>& a = da.b;
    real* sm = reinterpret_cast<real*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = a.N, E = 4 * N;
    const DenseLayout lay = dense_layout(N);
    const int T = lay.T, GS = lay.GS;
    DenseCtx<real> c{a};
    c.tid = tid; c.lane = lane; c.N = N; c.E = E; c.T = T; c.GS = GS;
    c.Ht = sm + lay.Ht; c.Lt = sm + lay.Lt;
    real* tiles = sm + lay.tiles;               // condensing / roll-out: the OCP's stage tiles (overlay Ht/Lt)
    real* Gc = sm + lay.Gc;
    real* evc = sm + lay.evc;
    real* sq = sm + lay.sq;                     // sqrt of the stage / terminal state weights
    real* small = sm + lay.sml;                 // wv(16) xp(16) red(16) control words
    real* red = small + 32;
    int* ctl = reinterpret_cast<int*>(small + 48);
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(small + 56);
    unsigned mphase = 0;                        // parity of the next TMA completion on mbar
    real* dxs = sm + lay.dxs;                   // state increments of the roll-out [(N+1)][13]
    real* v = sm + lay.vec;
    c.f = v; c.ubar = v + E; c.ucur = v + 2 * E; c.tl = v + 3 * E; c.tu = v + 4 * E; c.ll = v + 5 * E; c.lu = v + 6 * E;
    c.cl = v + 7 * E; c.cu = v + 8 * E; c.ua = v + 9 * E; c.usol = v + 10 * E; c.rt = v + 11 * E; c.dR = v + 12 * E;
    c.tv = v + 13 * E; c.itl = v + 14 * E; c.itu = v + 15 * E; c.ill = v + 16 * E; c.ilu = v + 17 * E;
    c.fx = c.cl; c.fv = c.cu;
    {   // tile owned by this thread
        int i = 0;
        while ((i + 1) * (i + 2) / 2 <= tid) ++i;
        c.ti = i; c.tj = tid - i * (i + 1) / 2;
    }
    const int ti = c.ti, tj = c.tj;
    {   // column-major map of the factorisation: column cc owns threads S(cc) .. S(cc) + N - cc (the last one = right-hand side)
        int cc = 0, start = 0;
        while (cc < N && start + (N - cc + 1) <= tid) { start += N - cc + 1; ++cc; }
        c.fj = cc < N ? cc : -1;
        c.fi = cc + (tid - start);
    }
    const int count = da.hard_list ? *da.hard_count : a.B;
    const real lb = a.lb, ub = a.ub;
    if (tid < NX) { sq[tid] = sqrt(a.Qd[tid]); sq[16 + tid] = sqrt(a.QNd[tid]); }
    if (tid == 0) mbar_init(mbar, 1);
    c.cbar = reinterpret_cast<unsigned long long*>(sm + lay.cbar);
    c.smbase = sm;
    c.fgen = 0;
    if (tid == 0) for (int k = 0; k < N; ++k) flag_init(c.cbar + k);      // one thread: compute-sanitizer loses mbarrier.init issued by several lanes at once
    const unsigned tile_bytes = (unsigned)(N * WT * sizeof(real));
    // condensing roles: thread t < T accumulates tile t of H; thread DN_THREADS-1-c carries impulse-response column c
    // (c < E) or the free response (c == E) through the stages - the LAST warps, whose tiles join the sum last, so the
    // propagation of chunk i+1 overlaps the tile accumulation of chunk i
    const int cidx = DN_THREADS - 1 - tid;
    const bool colthr = cidx <= E;
    // position of input column c = 4 blk + e inside a row of the impulse-response block.  QMPC_DENSE_GPLANES: two planes, entries
    // e = 0, 1 of every block contiguous in the first and e = 2, 3 in the second, so the 16-byte loads of a warp whose lanes
    // walk over the blocks fall into half as many 128-byte wavefronts as with the blocks' four entries side by side
    auto gcol = [GS](int c) -> int {
#if QMPC_DENSE_GPLANES
        return ((c >> 2) << 1) + (c & 1) + ((c >> 1) & 1) * (GS / 2);
#else
        (void)GS;
        return c;
#endif
    };
    const int nch = (N + DN_CH - 1) / DN_CH;
    enum { T_FIXED, T_ADJ, T_PRED, T_GRAD, T_DONE };
    __syncthreads();

    int item = blockIdx.x, qslot = 2;
    while (item < count) {
        // next item: fetched now, read after this item's last barrier (two alternating slots: the next write happens while
        // slower threads may still be reading the previous one)
        if (tid == 0) ctl[qslot] = da.next_item ? (int)gridDim.x + atomicAdd(da.next_item, 1) : item + (int)gridDim.x;
        const int ocp = da.hard_list ? da.hard_list[item] : item;
        if (a.timeline && tid == 0) a.timeline[2 * ocp] = global_ns();
        DPROF_DECL;
        const real* Wv = a.W + (size_t)ocp * N * WT;
        const double* x0 = a.x0 + (size_t)ocp * NX;
        const double* yref = a.yref + (size_t)ocp * N * NY;
        const double* yref_e = a.yref_e + (size_t)ocp * NX;
        double* xit = a.xit + (size_t)ocp * (N + 1) * NX;
        double* uit = a.uit + (size_t)ocp * N * NU;
        unsigned char* actset = a.act + (size_t)ocp * E;

        // ---- condensing: H = Rbar + sum_k G_k' Q_k G_k, f = Rbar (ubar - uref) + sum_k G_k' Q_k (free response + iterate - ref)
        if (tid == 0) {                          // every generic access to the overlay region ended at the last barrier
            fence_proxy_async();
            mbar_expect(mbar, tile_bytes);
            bulk_g2s(tiles, Wv, tile_bytes, mbar);
        }
        for (int idx = NX + tid; idx < (N + 1) * NX; idx += DN_THREADS) {     // iterate minus reference, stages 1..N
            const int k = idx / NX, r = idx - k * NX;
            dxs[idx] = real(xit[idx] - (k < N ? yref[(size_t)k * NY + r] : yref_e[r]));
        }
        real g[NX];
#pragma unroll
        for (int r = 0; r < NX; ++r) g[r] = cidx == E ? real(x0[r] - xit[r]) : real(0);
        if (tid < E) {
            const real ub_ = real(uit[tid]);
            c.ubar[tid] = ub_;
            c.f[tid] = a.Rd[tid & 3] * (ub_ - real(yref[(size_t)(tid >> 2) * NY + NX + (tid & 3)]));
        }
        real acc[16];
#pragma unroll
        for (int t = 0; t < 16; ++t) acc[t] = 0;
        real fc = 0;
        // one chunk of the column propagation: stages ch*DN_CH ..., results into buffer ch & 1
        auto propagate = [&](int ch) {
            real* Gb = Gc + (ch & 1) * (DN_CH * 13 * GS);
            real* eb = evc + (ch & 1) * (DN_CH * 16);
            for (int kk = 0; kk < DN_CH; ++kk) {
                const int k = ch * DN_CH + kk;
                if (k >= N) break;
                const int blk = cidx >> 2;               // stage at which input column cidx enters (E >> 2 == N: never)
                if (cidx < E && blk > k) continue;
                const real* tile = tiles + k * WT;
                const real* sqk = sq + ((k + 1 < N) ? 0 : 16);
                if (cidx < E && blk == k) {
#pragma unroll
                    for (int r = 0; r < NX; ++r) g[r] = tile[r * WR + (cidx & 3)];
                } else {
                    real gn[NX];
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        real s0 = r < 3 ? g[r] : real(0), s1 = 0;
#pragma unroll
                        for (int s_ = 0; s_ < 10; s_ += 2) {
                            real t0, t1;
                            ld2(tile + r * WR + 4 + s_, t0, t1);
                            s0 = fma(t0, g[3 + s_], s0); s1 = fma(t1, g[4 + s_], s1);
                        }
                        gn[r] = s0 + s1;
                    }
                    if (cidx == E) {
#pragma unroll
                        for (int r = 0; r < NX; ++r) gn[r] += tile[r * WR + 14];
                    }
#pragma unroll
                    for (int r = 0; r < NX; ++r) g[r] = gn[r];
                }
                if (cidx < E) {
#pragma unroll
                    for (int r = 0; r < NX; ++r) Gb[(kk * 13 + r) * GS + gcol(cidx)] = sqk[r] * g[r];
                } else {
#pragma unroll
                    for (int r = 0; r < NX; ++r) eb[kk * 16 + r] = sqk[r] * (g[r] + dxs[(k + 1) * NX + r]);
                }
            }
        };
        __syncthreads();                        // dxs is complete (the free-response thread reads it)
        bulk_wait_block(mbar, mphase); mphase ^= 1;
        if (colthr) propagate(0);
        __syncthreads();
        for (int ch = 0; ch < nch; ++ch) {
            if (colthr && ch + 1 < nch) propagate(ch + 1);
            const real* Gb = Gc + (ch & 1) * (DN_CH * 13 * GS);
            const real* eb = evc + (ch & 1) * (DN_CH * 16);
            if (tid < T) {                      // H tile += (sqrt(Q) G_i)' (sqrt(Q) G_j) over the stages of the chunk
                for (int kk = 0; kk < DN_CH; ++kk) {
                    const int k = ch * DN_CH + kk;
                    if (k >= N) break;
                    if (ti > k) continue;
                    const real* Gk = Gb + kk * 13 * GS;
#pragma unroll
                    for (int r = 0; r < NX; ++r) {
                        real gi[4], gj[4];
#if QMPC_DENSE_GPLANES
                        ld2(Gk + r * GS + 2 * ti, gi[0], gi[1]); ld2(Gk + r * GS + GS / 2 + 2 * ti, gi[2], gi[3]);
                        ld2(Gk + r * GS + 2 * tj, gj[0], gj[1]); ld2(Gk + r * GS + GS / 2 + 2 * tj, gj[2], gj[3]);
#else
                        ld2(Gk + r * GS + 4 * ti, gi[0], gi[1]); ld2(Gk + r * GS + 4 * ti + 2, gi[2], gi[3]);
                        ld2(Gk + r * GS + 4 * tj, gj[0], gj[1]); ld2(Gk + r * GS + 4 * tj + 2, gj[2], gj[3]);
#endif
#pragma unroll
                        for (int p = 0; p < 4; ++p)
#pragma unroll
                            for (int q = 0; q < 4; ++q) acc[p * 4 + q] = fma(gi[p], gj[q], acc[p * 4 + q]);
                    }
                }
            }
            if (tid < E) {                      // gradient entry of input tid
                for (int kk = 0; kk < DN_CH; ++kk) {
                    const int k = ch * DN_CH + kk;
                    if (k >= N) break;
                    if ((tid >> 2) > k) continue;
#pragma unroll
                    for (int r = 0; r < NX; ++r) fc = fma(Gb[(kk * 13 + r) * GS + gcol(tid)], eb[kk * 16 + r], fc);
                }
            }
            __syncthreads();                    // buffer (ch+1)&1 is complete; nobody reads buffer ch&1 any more
        }
        // every read of the overlay region ended at the barrier above: Ht may be written
        if (tid < T) {
            if (ti == tj) {
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[q * 5] += a.Rd[q];
            }
            real* o = c.Ht + tid * TS;
#pragma unroll
            for (int t = 0; t < 16; t += 2) st2(o + t, acc[t], acc[t + 1]);
        }
        if (tid < E) c.f[tid] += fc;
        // ---- box-QP: warp 0 drives (element-wise work, triangular solves, decisions); the CTA factors and multiplies.
        // Start: active-set rounds from the guess the screening kernel ended on (a round costs a quarter of a Riccati
        // round here), the IPM from the box centre if there is no guess or the rounds do not settle.
        int it = 0, rounds = 0, status = QMPC_STATUS_MAXITER_;
        bool exact = false, refine = a.max_refine > 0, ipm_started = false;
        int rounds_left = 0, prev_changed = 1 << 30, best_changed = 1 << 28, round_no = 0, attempts = 0;
        ActiveSetHistory hist;              // warp 0: fingerprints of the active sets of this attempt (cycle detection)
        hist.init(small + 57);              // 6 x 8 bytes of the scratch block
        if (warp == 0) {
            int known = a.dense_warm_rounds > 0 && da.hard_list != nullptr;
            DN_FOR_E(e) { const unsigned char fl = actset[e]; if (fl > 2) known = 0; c.fx[e] = real(fl <= 2 ? fl : 0); }
            known = warp_max(int(!known)) == 0;
            if (known) {
                DN_FOR_E(e) c.fv[e] = c.fx[e] == real(1) ? lb - c.ubar[e] : (c.fx[e] == real(2) ? ub - c.ubar[e] : real(0));
                rounds_left = a.dense_warm_rounds;
                rounds = a.rounds[ocp];              // rounds already spent in the screening kernel
            } else {
                DN_FOR_E(e) c.usol[e] = real(0.5) * (lb + ub) - c.ubar[e];
            }
            if (lane == 0) ctl[0] = known ? T_FIXED : T_GRAD;
        }
        __syncthreads();
        DPROF(0);
        real target = refine ? a.mu_switch : a.mu_tol, mu = 0, resfac = 1;
        const real inv2E = real(1) / real(2 * E);
        int trip = T_GRAD;
        while (true) {
            trip = ctl[0];
            if (trip == T_DONE) break;
            DPROF(5);
            // (1) products with H
            if (trip == T_GRAD || trip == T_ADJ) { c.matvec(c.usol); __syncthreads(); }
            else if (trip == T_FIXED) { c.matvec(c.fv); __syncthreads(); }
            DPROF(1);
            // (2) right-hand side, factorisation
            if (trip == T_FIXED || trip == T_PRED) {
                if (warp == 0) {
                    if (trip == T_FIXED) {
                        DN_FOR_E(e) c.rt[e] = c.fx[e] != real(0) ? c.fv[e] : -c.f[e] - c.tv[e];
                    } else {
                        DN_FOR_E(e) {
                            const real itl = real(1) / c.tl[e], itu = real(1) / c.tu[e];
                            const real ll = c.ll[e], lu = c.lu[e];
                            c.itl[e] = itl; c.itu[e] = itu; c.ill[e] = real(1) / ll; c.ilu[e] = real(1) / lu;
                            const real d = ll * itl + lu * itu;
                            c.dR[e] = d;
                            c.rt[e] = -c.f[e] + d * (c.ucur[e] - c.ubar[e]);
                        }
                    }
                }
                __syncthreads();
                DPROF(7);
#if QMPC_DENSE_FACTOR == 2
                c.factor_rl1(trip == T_FIXED);
#elif QMPC_DENSE_FACTOR == 1
                c.factor_cols(trip == T_FIXED);
#else
                c.factor(trip == T_FIXED);
#endif
                c.scale_for_solves();
            }
            DPROF(2);
            // (3) warp 0: solves, step logic, next trip
            if (warp == 0) {
                int next = T_DONE;
                if (trip == T_GRAD) {
                    real gs = 0;
                    DN_FOR_E(e) gs += fabs(c.tv[e] + c.f[e]);
                    gs = warp_sum(gs) / real(E);
                    const real lam0 = rfinite(gs) ? fmin(fmax(a.lam0_scale * gs, a.lam0_min), a.lam0_max) : a.lam0_min;
                    DN_FOR_E(e) {
                        const real u0 = real(0.5) * (lb + ub);
                        c.ucur[e] = u0; c.tl[e] = u0 - lb; c.tu[e] = ub - u0; c.ll[e] = lam0; c.lu[e] = lam0;
                    }
                    ipm_started = true;
                    next = T_PRED;
                } else if (trip == T_FIXED) {
                    c.solve(c.rt, c.usol, true);
                    DPROF(8);
                    next = T_ADJ;
                } else if (trip == T_ADJ) {
                    ++rounds;
                    int changed = 0;
                    unsigned long long fp = 0;
                    DN_FOR_E(e) {
                        const real fxe = c.fx[e], un = c.ubar[e] + c.usol[e], gr = c.tv[e] + c.f[e];
                        real fn = fxe;
                        if (fxe == real(1)) { if (gr < -a.refine_gtol) fn = 0; }
                        else if (fxe == real(2)) { if (gr > a.refine_gtol) fn = 0; }
                        else if (un < lb) fn = 1;
                        else if (un > ub) fn = 2;
                        if (fn != fxe) { ++changed; c.fx[e] = fn; }
                        c.fv[e] = fn == real(1) ? lb - c.ubar[e] : (fn == real(2) ? ub - c.ubar[e] : real(0));
                        fp += active_set_term(e, fn);
                    }
                    changed = warp_sum(changed);
                    fp = warp_sum(fp);
                    // the primal-dual active-set iteration is a deterministic map of the active set: meeting a set again
                    // means it cycles (period 3-4 in practice) and will never settle from this start
                    const bool cycling = hist.seen_then_push(fp, lane) && changed;
                    ++round_no;
#ifdef QMPC_EMU_TRACE
                    if (lane == 0) {
                        int np_ = 0; real gmin = 1e30;
                        for (int e = 0; e < E; ++e) if (c.fx[e] != real(0)) ++np_;
                        printf("  [trace ocp %d] round %d (ipm_started %d it %d): changed %d pinned %d cycling %d\n", ocp, round_no, (int)ipm_started, it, changed, np_, (int)cycling);
                    }
#endif
                    if (!changed) { exact = true; status = QMPC_STATUS_OK_; next = T_DONE; }
                    else if (--rounds_left > 0 && !cycling && !(ipm_started && round_no >= 2 && changed > 2 * best_changed + 2) &&
                             !((!ipm_started || a.post_bail) && round_no >= 3 && changed >= prev_changed)) {
                        // after the IPM (fp64) the rounds only give up on a proven cycle or when the change count runs away
                        // from its best value (a diverging iteration wanders for all its rounds; the sharper restart settles)
                        prev_changed = changed; best_changed = changed < best_changed ? changed : best_changed; next = T_FIXED;
                    }
                    else if (!ipm_started) {     // the warm rounds did not settle: IPM from the box centre
                        DN_FOR_E(e) c.usol[e] = real(0.5) * (lb + ub) - c.ubar[e];
                        next = T_GRAD;
                    } else if (++attempts < 3) {
                        // one more attempt from a 100x sharper IPM point, then a last one from the IPM point at mu_tol (as
                        // qmpc_ipm_kernel).  If that does not settle either, the IPM point is returned with status MAXITER
                        // and flags 255, never as status 0: it is not the minimiser (1e-9..2e-8 off at N = 20 with
                        // refine_max_rounds = 1, while its rounded active set already matched the exact one)
                        target = attempts < 2 ? target * real(1e-2) : a.mu_tol;
                        next = T_PRED;
                    }
                } else if (trip == T_PRED) {
                    DPROF(6);
                    c.solve(c.rt, c.usol, true);
                    DPROF(3);
                    // predictor: step lengths (as reciprocals: alpha = 1 / max ratio), centring parameter
                    real rpm = 1, rdm = 1;
                    DN_FOR_E(e) {
                        const real itl = c.itl[e], itu = c.itu[e], ll = c.ll[e], lu = c.lu[e];
                        const real us = c.usol[e];
                        const real du = c.ubar[e] + us - c.ucur[e];
                        const real dl = -ll - ll * itl * du;
                        const real dv = -lu + lu * itu * du;
                        c.ua[e] = us;
                        c.cl[e] = du * dl; c.cu[e] = -du * dv;
                        c.rt[e] = dl; c.tv[e] = dv;
                        rpm = fmax(rpm, fmax(-du * itl, du * itu));
                        rdm = fmax(rdm, fmax(-dl * c.ill[e], -dv * c.ilu[e]));
                    }
                    const real apa = real(1) / warp_max(rpm), ada = real(1) / warp_max(rdm);
                    real s = 0;
                    DN_FOR_E(e) {
                        const real du = c.ubar[e] + c.ua[e] - c.ucur[e];
                        s += (c.ll[e] + ada * c.rt[e]) * (c.tl[e] + apa * du) + (c.lu[e] + ada * c.tv[e]) * (c.tu[e] - apa * du);
                    }
                    const real muaff = warp_sum(s) * inv2E;
                    real sigma = muaff / mu; sigma = sigma * sigma * sigma;
                    // corrector (increment on the predictor); a blocked Mehrotra step is redone once as a centring step
                    real so = 1;
                    for (int cpass = 0; cpass < 2; ++cpass) {
                        const real smu = sigma * mu;
                        DN_FOR_E(e) c.rt[e] = (smu - so * c.cl[e]) * c.itl[e] - (smu - so * c.cu[e]) * c.itu[e];
                        __syncwarp();
                        DPROF(6);
                        c.solve(c.rt, c.usol, false);
                        DPROF(3);
                        real rpx = real(1e-30), rdx = real(1e-30);
                        DN_FOR_E(e) {
                            const real itl = c.itl[e], itu = c.itu[e], ll = c.ll[e], lu = c.lu[e];
                            const real du = c.ubar[e] + c.ua[e] + c.usol[e] - c.ucur[e];
                            const real dl = (smu - so * c.cl[e]) * itl - ll - ll * itl * du;
                            const real dv = (smu - so * c.cu[e]) * itu - lu + lu * itu * du;
                            c.usol[e] = du; c.rt[e] = dl; c.tv[e] = dv;
                            rpx = fmax(rpx, fmax(-du * itl, du * itu));
                            rdx = fmax(rdx, fmax(-dl * c.ill[e], -dv * c.ilu[e]));
                        }
                        real ap = real(1) / warp_max(rpx), ad = real(1) / warp_max(rdx);
                        if (cpass == 0 && fmin(ap, ad) < real(0.5)) { so = 0; sigma = fmax(sigma, real(0.5)); continue; }
                        ap = fmin(real(1), real(0.995) * ap); ad = fmin(real(1), real(0.995) * ad);
                        DN_FOR_E(e) {
                            const real du = ap * c.usol[e];
                            c.ucur[e] += du; c.tl[e] += du; c.tu[e] -= du;
                            c.ll[e] += ad * c.rt[e];
                            c.lu[e] += ad * c.tv[e];
                        }
                        resfac *= real(1) - fmin(ap, ad);
                        ++it;
#ifdef QMPC_EMU_TRACE
                        if (lane == 0) printf("  [trace ocp %d] ipm it %d: mu %.3e sigma %.3e ap %.4f ad %.4f resfac %.3e cpass %d\n", ocp, it, (double)mu, (double)sigma, (double)ap, (double)ad, (double)resfac, cpass);
#endif
                        break;
                    }
                    next = T_PRED;
                }
                if (next == T_PRED) {           // complementarity, convergence / hand-over test
                    __syncwarp();
                    real s = 0;
                    DN_FOR_E(e) s += c.ll[e] * c.tl[e] + c.lu[e] * c.tu[e];
                    mu = warp_sum(s) * inv2E;
                    if (!rfinite(mu)) { status = QMPC_STATUS_NAN_; next = T_DONE; }
                    else if (mu < target && resfac < (refine ? real(1e-3) : a.resfac_final)) {
                        if (refine) {
                            DN_FOR_E(e) {
                                const real fn = c.tl[e] < c.ll[e] ? real(1) : (c.tu[e] < c.lu[e] ? real(2) : real(0));
                                c.fx[e] = fn;
                                c.fv[e] = fn == real(1) ? lb - c.ubar[e] : (fn == real(2) ? ub - c.ubar[e] : real(0));
                            }
                            next = T_FIXED; rounds_left = a.max_refine; prev_changed = 1 << 30; best_changed = 1 << 28; round_no = 0; hist.clear();
                        } else { status = QMPC_STATUS_OK_; next = T_DONE; }
                    } else if (it >= iter_limit(a, ocp)) next = T_DONE;
                }
                __syncwarp();
                if (lane == 0) ctl[0] = next;
                DPROF(6);
            }
            __syncthreads();
        }
        // ---- result: new iterate, states re-rolled through the linearised dynamics.  Ht/Lt are dead: the stage tiles
        //      come back into the overlay region with one more TMA bulk copy while warp 0 finalises the inputs.
        if (tid == 0) {
            fence_proxy_async();
            mbar_expect(mbar, tile_bytes);
            bulk_g2s(tiles, Wv, tile_bytes, mbar);
        }
        if (warp == 0) {
            real chk = 0;
            DN_FOR_E(e) { const real un = exact ? c.usol[e] : c.ucur[e]; chk += un - un; }
            chk = warp_sum(chk);
            if (!(chk == real(0))) status = QMPC_STATUS_NAN_;
            const bool good = status != QMPC_STATUS_NAN_;
            if (lane == 0) ctl[1] = good ? 1 : 0;
            if (!good) {
                DN_FOR_E(e) actset[e] = 255;
                if (lane < 4) a.u0[(size_t)ocp * 4 + lane] = double(fmin(fmax(c.ubar[lane], lb), ub));
                if (lane == 0) { a.cost[ocp] = nan(""); a.status[ocp] = status; a.iters[ocp] = it; a.rounds[ocp] = rounds; }
            } else {
                DN_FOR_E(e) {
                    real un;
                    unsigned char fl;
                    if (exact) {
                        fl = c.fx[e] == real(1) ? 1 : (c.fx[e] == real(2) ? 2 : 0);
                        un = fl == 1 ? lb : (fl == 2 ? ub : c.ubar[e] + c.usol[e]);
                    } else {
                        un = fmin(fmax(c.ucur[e], lb), ub);
                        fl = status == QMPC_STATUS_OK_ ? (c.tl[e] < c.ll[e] ? 1 : (c.tu[e] < c.lu[e] ? 2 : 0)) : 255;
                    }
                    actset[e] = fl;
                    c.ucur[e] = un;
                    c.usol[e] = un - c.ubar[e];
                    uit[e] = double(un);
                }
                if (lane < 4) a.u0[(size_t)ocp * 4 + lane] = double(c.ucur[lane]);
            }
            // dx_{k+1} = A dx_k + B du_k + b_k: lane j < 13 owns row j of the stage tile and walks its 16 columns starting
            // at column j (rows are 128 B apart: the rotation keeps the lanes on different banks)
            real* wv = small;                   // [du(4), dx_3..12(10), 1, 0]
            real* xp = small + 16;              // dx_0..2 (the position columns of A are unit vectors)
            if (lane < NX) {
                const real d0 = real(x0[lane] - xit[lane]);
                if (lane < 3) xp[lane] = d0; else wv[lane + 1] = d0;
            } else if (lane == 14) wv[14] = 1;
            else if (lane == 15) wv[15] = 0;
            bulk_wait_warp(mbar, mphase);       // the tiles have landed (waited for on the NaN path too: the barrier is reused)
            if (good) {
                const int j = lane < NX ? lane : NX - 1;
                for (int k = 0; k < N; ++k) {
                    if (lane < 4) wv[lane] = c.usol[k * 4 + lane];
                    __syncwarp();
                    const real* tr = tiles + k * WT + j * WR;
                    real s0 = 0, s1 = 0, s2 = 0, s3 = 0;
#pragma unroll
                    for (int q = 0; q < 16; q += 4) {
                        const int c0 = (q + j) & 15, c1 = (q + 1 + j) & 15, c2 = (q + 2 + j) & 15, c3 = (q + 3 + j) & 15;
                        s0 = fma(tr[c0], wv[c0], s0); s1 = fma(tr[c1], wv[c1], s1);
                        s2 = fma(tr[c2], wv[c2], s2); s3 = fma(tr[c3], wv[c3], s3);
                    }
                    real accx = (s0 + s1) + (s2 + s3);
                    if (lane < 3) accx += xp[lane];
                    __syncwarp();
                    if (lane < NX) {
                        if (lane < 3) xp[lane] = accx; else wv[lane + 1] = accx;
                        dxs[(k + 1) * NX + lane] = accx;
                    }
                    __syncwarp();
                }
            }
        }
        mphase ^= 1;
        __syncthreads();
        DPROF(4);
        if (ctl[1]) {       // new states and objective, all threads
            real cs = 0;
            for (int idx = tid; idx < (N + 1) * NX; idx += DN_THREADS) {
                const int k = idx / NX, r = idx - k * NX;
                const double xnew = k == 0 ? x0[r] : xit[idx] + double(dxs[idx]);
                xit[idx] = xnew;
                const real w = k < N ? a.Qd[r] : a.QNd[r];
                const real e_ = real(xnew - (k < N ? yref[(size_t)k * NY + r] : yref_e[r]));
                cs += real(0.5) * w * e_ * e_;
            }
            if (tid < E) {
                const real e_ = real(double(c.ucur[tid]) - yref[(size_t)(tid >> 2) * NY + NX + (tid & 3)]);
                cs += real(0.5) * a.Rd[tid & 3] * e_ * e_;
            }
            cs = warp_sum(cs);
            if (lane == 0) red[warp] = cs;
            __syncthreads();
            if (tid == 0) {
                real tot = 0;
                for (int w = 0; w < DN_THREADS / 32; ++w) tot += red[w];
                a.cost[ocp] = double(tot); a.status[ocp] = status; a.iters[ocp] = it; a.rounds[ocp] = rounds;
            }
        }
        if (a.timeline && tid == 0) a.timeline[2 * ocp + 1] = global_ns();
#ifdef QMPC_DENSE_PROF
        if (tid == 0 && item < 3)
            printf("dense ocp %d it %d rounds %d | cycles: condense %lld | matvec %lld (%d) | factor %lld (%d) | rhs %lld (%d) | solves %lld (%d) | back-substitution of a round %lld (%d) | logic %lld | rollout %lld | loop-top %lld | total %lld\n",
                   ocp, it, rounds, pf_acc[0], pf_acc[1], pf_n[1], pf_acc[2], pf_n[2], pf_acc[7], pf_n[7], pf_acc[3], pf_n[3], pf_acc[8], pf_n[8], pf_acc[6], pf_acc[4], pf_acc[5], clock64() - pf_t0);
#endif
        __syncthreads();
        item = ctl[qslot];
        qslot ^= 1;
    }
}

}  // namespace qmpc
