// capi.cu — C-ABI of libqmpc.so (include/qmpc.h): handle management and kernel launches.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC capi.cu -o libqmpc.so
#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/qmpc.h"
#include "aux_kernels.cuh"
#include "host_params.h"
#include "mpc_kernels.cuh"
#include "mpc_kernels_dense.cuh"
#include "rgp_kernels.cuh"

using namespace qmpc;

namespace {

thread_local std::string g_err;
std::atomic<long long> g_launches{0};

int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}

#define CU_TRY(expr)                                                                                   \
    do {                                                                                               \
        cudaError_t e_ = (expr);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(QMPC_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));            \
    } while (0)

#define LAUNCH_CHECK()                                                                                 \
    do {                                                                                               \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                            \
        cudaError_t e_ = cudaGetLastError();                                                           \
        if (e_ != cudaSuccess) return fail(QMPC_ERR_CUDA, std::string("launch: ") + cudaGetErrorString(e_)); \
    } while (0)

inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }
inline int cdiv(long long a, long long b) { return int((a + b - 1) / b); }

#ifndef QMPC_IPM_WARPS
#define QMPC_IPM_WARPS 1      // one OCP per CTA: a finished warp frees its SM slot at once (IPM iteration counts vary)
#endif
constexpr int IPM_WARPS = QMPC_IPM_WARPS;
constexpr int RGP_WARPS = 4;

}  // namespace

struct qmpc_solver {
    qmpc_config cfg;
    double dt;
    size_t rsz;                       // sizeof(real)
    double *x0 = nullptr, *yref = nullptr, *yref_e = nullptr, *alpha = nullptr, *xit = nullptr, *uit = nullptr;
    double *u0 = nullptr, *cost = nullptr, *gpX = nullptr, *xt = nullptr, *yt = nullptr;
    double gp_grid[6] = {0, 0, 0, 0, 0, 0};   // per axis {first basis point, spacing} of an equispaced grid (spacing 0: general path)
    int *status = nullptr, *iters = nullptr, *rounds = nullptr;
    unsigned char* act = nullptr;     // [B][4N] active sets remembered for the warm start
    void *W = nullptr, *fac = nullptr;
    int* fail_streak = nullptr;       // [B] consecutive failed solves per vehicle
    int* hard = nullptr;              // [B + 1] list of OCPs handed from the screening kernel to the dense kernel, then the count
    int dense_grid = 0;
    long long* timeline = nullptr;    // [B][2] per-OCP start/end stamps when enabled
    int variant = 2;                  // host_params.h solver_variant(): 1 Riccati kernel alone, 2 Riccati screening + dense kernel
    bool reset_failed = true;         // qmpc_config::reset_on_fail
    int parity = 0;                   // which of the two unsettled counters this solve writes
    const double* x0_src = nullptr;   // where the next solve reads x0 / alpha from (own buffers or bound ones)
    const double* alpha_src = nullptr;
    int alpha_stride = 0;
    ModelParams<double> mp64;
    bool timing = false;              // cudaEvents around the two solve kernels (bench roofline leg only)
    std::vector<cudaEvent_t> ev;      // triples: before linearize, before ipm, after ipm
    std::vector<cudaEvent_t> ev_mid;  // between the screening and the dense kernel (one per timed solve)
    bool solved = false;              // a solve has been queued: the stage tiles W hold data (qmpc_eval_sens_x0)
    long long epoch = 0;              // qmpc_get_sens_epoch: bumped whenever the tiles or the active set may change
    double w_solved[NY] = {}, we_solved[NX] = {};   // the weights the last solve ran with (cfg holds those of the next solve)
};

struct qrgp_model {
    int B, M, device;
    double *X = nullptr, *theta = nullptr, *Kx = nullptr, *Kx_inv = nullptr;
    double *mu = nullptr, *C = nullptr, *alpha = nullptr, *xt = nullptr, *yt = nullptr;
    double* part = nullptr;           // shared-swarm mode: per-CTA partial sums [3][part_ctas][M*M+M]
    int sms = 148, part_ctas = 0, acc_warps = 0;
    bool pushed = false;              // a regress has produced alpha since create / set_state: the reference pushes the RGP
                                      // means into the solver only after its first regress (quad_opt.py:101,402-404)
};

struct qrgpl_model {
    int n, M, device;
    double *X = nullptr, *mu_g = nullptr, *C_g = nullptr, *mu_eta = nullptr, *C_eta = nullptr, *C_g_eta = nullptr, *Kx_inv = nullptr;
    int* status = nullptr;
};

extern "C" {

const char* qmpc_last_error(void) { return g_err.c_str(); }
int qmpc_version(void) { return 100; }
long long qmpc_launch_count(void) { return g_launches.load(); }

// ------------------------------------------------------------------------------------------- solver

int qmpc_destroy(qmpc_handle_t h);

int qmpc_create(const qmpc_config* cfg, qmpc_handle_t* out)
{
    if (!cfg || !out) return fail(QMPC_ERR_ARG, "null argument");
    if (cfg->batch < 1 || cfg->n_nodes < 1 || cfg->n_nodes > 256) return fail(QMPC_ERR_ARG, "batch/n_nodes out of range");
    if (cfg->n_basis < 0 || cfg->n_basis > 128) return fail(QMPC_ERR_ARG, "n_basis must be in [0,128]");
    if (cfg->precision != 64 && cfg->precision != 32 && cfg->precision != 0) return fail(QMPC_ERR_ARG, "precision must be 64 or 32");
    if (cfg->precision == 32 && cfg->n_nodes > QMPC_FP32_MAX_NODES)
        return fail(QMPC_ERR_ARG, "fp32 handles (precision 32) take n_nodes <= QMPC_FP32_MAX_NODES (64)");
    if (cfg->n_basis > 0 && !cfg->gp_X) return fail(QMPC_ERR_ARG, "gp_X is NULL with n_basis > 0");
    // finite bounds only: the IPM starts from the box centre 0.5 (lbu + ubu)
    if (!(cfg->t_horizon > 0) || !(cfg->ubu > cfg->lbu) || !std::isfinite(cfg->lbu) || !std::isfinite(cfg->ubu))
        return fail(QMPC_ERR_ARG, "t_horizon / bounds invalid");
    if (cfg->solver_variant < 0 || cfg->solver_variant > 2) return fail(QMPC_ERR_ARG, "solver_variant must be 0, 1 or 2");
    if (cfg->solver_variant == 2 && (cfg->precision == 32 || cfg->n_nodes > DN_MAX_N))
        return fail(QMPC_ERR_ARG, "solver_variant 2 (screening + dense) needs fp64 and n_nodes <= 21");
    CU_TRY(cudaSetDevice(cfg->device));
    // every early return below releases what was allocated so far
    std::unique_ptr<qmpc_solver, int (*)(qmpc_handle_t)> guard(new qmpc_solver(), qmpc_destroy);
    qmpc_solver* h = guard.get();
    h->cfg = *cfg;
    if (h->cfg.precision == 0) h->cfg.precision = 64;
    h->cfg.gp_X = nullptr;
    h->dt = cfg_dt(*cfg);
    h->rsz = h->cfg.precision == 64 ? 8 : 4;
    h->reset_failed = cfg->reset_on_fail >= 0;
    const size_t B = cfg->batch, N = cfg->n_nodes, M = cfg->n_basis;
    fill_model(*cfg, h->mp64);
#define ALLOC(p, n) CU_TRY(cudaMalloc(reinterpret_cast<void**>(&(p)), (n)))
    ALLOC(h->x0, B * NX * 8); ALLOC(h->yref, B * N * NY * 8); ALLOC(h->yref_e, B * NX * 8);
    ALLOC(h->alpha, B * 3 * (M ? M : 1) * 8); ALLOC(h->xit, B * (N + 1) * NX * 8); ALLOC(h->uit, B * N * NU * 8);
    ALLOC(h->u0, B * NU * 8); ALLOC(h->cost, B * 8); ALLOC(h->status, B * 4); ALLOC(h->iters, B * 4);
    ALLOC(h->xt, B * 3 * 8); ALLOC(h->yt, B * 3 * 8); ALLOC(h->rounds, B * 4); ALLOC(h->act, B * N * NU);
    ALLOC(h->fail_streak, B * 4);
    ALLOC(h->W, (B * N + 1) * WT * h->rsz); ALLOC(h->fac, B * N * FAC * h->rsz);
    ALLOC(h->gpX, 3 * (M ? M : 1) * 8);
#undef ALLOC
    CU_TRY(cudaMemset(h->x0, 0, B * NX * 8)); CU_TRY(cudaMemset(h->yref, 0, B * N * NY * 8));
    CU_TRY(cudaMemset(h->yref_e, 0, B * NX * 8)); CU_TRY(cudaMemset(h->alpha, 0, B * 3 * (M ? M : 1) * 8));
    CU_TRY(cudaMemset(h->xit, 0, B * (N + 1) * NX * 8)); CU_TRY(cudaMemset(h->uit, 0, B * N * NU * 8));
    CU_TRY(cudaMemset(h->u0, 0, B * NU * 8)); CU_TRY(cudaMemset(h->cost, 0, B * 8));
    CU_TRY(cudaMemset(h->status, 0, B * 4)); CU_TRY(cudaMemset(h->iters, 0, B * 4));
    CU_TRY(cudaMemset(h->rounds, 0, B * 4)); CU_TRY(cudaMemset(h->act, 255, B * N * NU));
    CU_TRY(cudaMemset(h->fail_streak, 0, B * 4));
    if (M) CU_TRY(cudaMemcpy(h->gpX, cfg->gp_X, 3 * M * 8, cudaMemcpyHostToDevice));
    gp_grid_detect(M ? cfg->gp_X : nullptr, M, h->gp_grid);
    h->x0_src = h->x0; h->alpha_src = h->alpha; h->alpha_stride = 3 * (int)M;
    const size_t smem64 = (size_t)IPM_WARPS * ipm_smem_reals((int)N, true, true) * 8, smem32 = (size_t)IPM_WARPS * ipm_smem_reals((int)N, true, false) * 4;
    if (smem64 > 220 * 1024) return fail(QMPC_ERR_ARG, "n_nodes too large for the shared-memory plan");
    CU_TRY(cudaFuncSetAttribute(qmpc_ipm_kernel<double, IPM_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem64));
    CU_TRY(cudaFuncSetAttribute(qmpc_ipm_kernel<float, IPM_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem32));
    CU_TRY(cudaFuncSetAttribute(qmpc_sens_kernel<double, IPM_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                IPM_WARPS * ipm_smem_reals((int)N, false, true) * 8));
    CU_TRY(cudaFuncSetAttribute(qmpc_adjoint_kernel<double, IPM_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                IPM_WARPS * ipm_smem_reals((int)N, false, true) * 8));
    CU_TRY(cudaFuncSetAttribute(qmpc_adjoint_kernel<double, IPM_WARPS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                IPM_WARPS * ipm_smem_reals((int)N, false, true) * 8));
    CU_TRY(cudaFuncSetAttribute(qmpc_jvp_kernel<double, IPM_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                IPM_WARPS * ipm_smem_reals((int)N, false, true) * 8));
    h->variant = solver_variant(h->cfg, DN_MAX_N);
    if (h->variant == 2) {
        const int smemd = dense_layout((int)N).total * 8;
        CU_TRY(cudaMalloc(reinterpret_cast<void**>(&h->hard), (B + 4) * sizeof(int)));      // list, count, work-queue counter, unsettled x2
        CU_TRY(cudaMemset(h->hard, 0, (B + 4) * sizeof(int)));
        CU_TRY(cudaFuncSetAttribute(qmpc_dense_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, smemd));
        int per_sm = 0, sms = 0;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, qmpc_dense_kernel<double>, DN_THREADS, smemd));
        CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device));
        // persistent CTAs taking items of the hard list from a work queue: 10-15 % of the vehicles are on it in steady
        // state and up to 40 % in a start-up transient; a third of the batch (at most one resident wave) measured best
        // (profiles/r02_policy_ab.txt), more only queues empty CTAs behind other streams' kernels
        const size_t want = cfg->dense_grid > 0 ? (size_t)cfg->dense_grid : std::max<size_t>(32, B / 3);
        h->dense_grid = (int)std::min<size_t>(std::min<size_t>(B, want), (size_t)std::max(1, per_sm) * sms);
    }
    CU_TRY(cudaDeviceSynchronize());
    *out = guard.release();
    return QMPC_OK;
}

int qmpc_destroy(qmpc_handle_t h)
{
    if (!h) return QMPC_OK;
    cudaSetDevice(h->cfg.device);
    void* ps[] = {h->x0, h->yref, h->yref_e, h->alpha, h->xit, h->uit, h->u0, h->cost, h->status, h->iters,
                  h->W, h->fac, h->gpX, h->xt, h->yt, h->rounds, h->act, h->timeline, h->hard, h->fail_streak};
    for (void* p : ps) if (p) cudaFree(p);
    for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_mid) cudaEventDestroy(e);
    delete h;
    return QMPC_OK;
}

static int copy_dd(void* dst, const void* src, size_t bytes, void* stream)
{
    if (!dst || !src) return fail(QMPC_ERR_ARG, "null pointer");
    CU_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, S(stream)));
    return QMPC_OK;
}

int qmpc_set_yref(qmpc_handle_t h, const double* yref, const double* yref_e, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    const size_t B = h->cfg.batch, N = h->cfg.n_nodes;
    int rc = copy_dd(h->yref, yref, B * N * NY * 8, stream);
    if (rc) return rc;
    return copy_dd(h->yref_e, yref_e, B * NX * 8, stream);
}

int qmpc_set_reference(qmpc_handle_t h, const double* x_ref, const double* u_ref, void* stream)
{
    if (!h || !x_ref) return fail(QMPC_ERR_ARG, "null argument");
    const int B = h->cfg.batch, N = h->cfg.n_nodes;
    set_reference_kernel<<<cdiv((long long)B * N * NY, 256), 256, 0, S(stream)>>>(B, N, x_ref, u_ref, 0.16, h->yref, h->yref_e);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qmpc_set_x0(qmpc_handle_t h, const double* x0, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    h->x0_src = h->x0;
    return copy_dd(h->x0, x0, (size_t)h->cfg.batch * NX * 8, stream);
}

int qmpc_set_params(qmpc_handle_t h, const double* mu, const double* Kx_inv, void* stream)
{
    if (!h || !mu || !Kx_inv) return fail(QMPC_ERR_ARG, "null argument");
    const int B = h->cfg.batch, M = h->cfg.n_basis;
    if (M == 0) return fail(QMPC_ERR_ARG, "solver was created without an RGP model (n_basis == 0)");
    qrgp_alpha_kernel<<<cdiv((long long)B * 3 * M, 128), 128, 0, S(stream)>>>(B, M, Kx_inv, mu, h->alpha);
    LAUNCH_CHECK();
    h->alpha_src = h->alpha; h->alpha_stride = 3 * M;
    return QMPC_OK;
}

int qmpc_set_alpha(qmpc_handle_t h, const double* alpha, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (h->cfg.n_basis == 0) return fail(QMPC_ERR_ARG, "solver was created without an RGP model (n_basis == 0)");
    h->alpha_src = h->alpha; h->alpha_stride = 3 * h->cfg.n_basis;
    return copy_dd(h->alpha, alpha, (size_t)h->cfg.batch * 3 * h->cfg.n_basis * 8, stream);
}

int qmpc_bind_alpha(qmpc_handle_t h, const double* alpha, int stride)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (h->cfg.n_basis == 0) return fail(QMPC_ERR_ARG, "solver was created without an RGP model (n_basis == 0)");
    if (alpha && stride != 0 && stride != 3 * h->cfg.n_basis) return fail(QMPC_ERR_ARG, "stride must be 0 (one shared model) or 3*n_basis");
    h->alpha_src = alpha ? alpha : h->alpha;
    h->alpha_stride = alpha ? stride : 3 * h->cfg.n_basis;
    return QMPC_OK;
}

int qmpc_set_weights(qmpc_handle_t h, const double* w_diag, const double* we_diag)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (!w_diag && !we_diag) return fail(QMPC_ERR_ARG, "w_diag and we_diag are both NULL");
    for (int i = 0; w_diag && i < NY; ++i) {
        if (!std::isfinite(w_diag[i]) || w_diag[i] < 0) return fail(QMPC_ERR_ARG, "w_diag entries must be finite and >= 0");
        // the Riccati and the dense factorisations need R positive definite
        if (i >= NX && !(w_diag[i] > 0)) return fail(QMPC_ERR_ARG, "the input weights w_diag[13..16] must be > 0");
    }
    for (int i = 0; we_diag && i < NX; ++i)
        if (!std::isfinite(we_diag[i]) || we_diag[i] < 0) return fail(QMPC_ERR_ARG, "we_diag entries must be finite and >= 0");
    if (w_diag) std::memcpy(h->cfg.w_diag, w_diag, sizeof(h->cfg.w_diag));
    if (we_diag) std::memcpy(h->cfg.we_diag, we_diag, sizeof(h->cfg.we_diag));
    return QMPC_OK;
}

int qmpc_set_iterate(qmpc_handle_t h, const double* x, const double* u, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    const size_t B = h->cfg.batch, N = h->cfg.n_nodes;
    int rc = copy_dd(h->xit, x, B * (N + 1) * NX * 8, stream);
    if (rc) return rc;
    CU_TRY(cudaMemsetAsync(h->status, 0, B * sizeof(int), S(stream)));      // an explicit iterate is never re-initialised
    CU_TRY(cudaMemsetAsync(h->fail_streak, 0, B * sizeof(int), S(stream)));
    return copy_dd(h->uit, u, B * N * NU * 8, stream);
}

int qmpc_get_iterate(qmpc_handle_t h, double* x, double* u, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    const size_t B = h->cfg.batch, N = h->cfg.n_nodes;
    int rc = copy_dd(x, h->xit, B * (N + 1) * NX * 8, stream);
    if (rc) return rc;
    return copy_dd(u, h->uit, B * N * NU * 8, stream);
}

}  // extern "C"

template <typename real>
static int solve_impl(qmpc_solver* h, void* stream)
{
    ++h->epoch;                     // qmpc_solve, qmpc_step(_dt) and qmpc_closed_loop_step all come through here
    std::memcpy(h->w_solved, h->cfg.w_diag, sizeof(h->w_solved));
    std::memcpy(h->we_solved, h->cfg.we_diag, sizeof(h->we_solved));
    const int B = h->cfg.batch, N = h->cfg.n_nodes;
    LinArgs<double, real> la;       // the linearisation always runs in fp64; fp32 handles store fp32 tiles (see LinArgs)
    fill_lin_args(h->cfg, la);
    la.xit = h->xit; la.uit = h->uit; la.yref = h->yref; la.alpha = h->alpha_src; la.alpha_stride = h->alpha_stride;
    la.gpX = h->gpX; la.W = static_cast<real*>(h->W);
    fill_gp_grid(h->gp_grid, la.mp);
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    if (h->timing && h->ev.size() < 3 * 8192) {
        CU_TRY(cudaEventCreate(&e0)); CU_TRY(cudaEventCreate(&e1)); CU_TRY(cudaEventCreate(&e2));
        h->ev.push_back(e0); h->ev.push_back(e1); h->ev.push_back(e2);
        CU_TRY(cudaEventRecord(e0, S(stream)));
    }
    if (h->reset_failed) {
        reset_failed_kernel<<<cdiv((long long)B * (N + 1), 256), 256, 0, S(stream)>>>(B, N, h->status, h->yref, h->yref_e, h->xit, h->uit, h->act, h->fail_streak);
        LAUNCH_CHECK();
    }
    qmpc_linearize_kernel<double, real><<<cdiv((long long)B * N, LIN_NB), LIN_THREADS, 0, S(stream)>>>(la);
    LAUNCH_CHECK();
    if (e1) CU_TRY(cudaEventRecord(e1, S(stream)));
    IpmArgs<real> ia;
    fill_ipm_args(h->cfg, ia);
    ia.x0 = h->x0_src; ia.yref = h->yref; ia.yref_e = h->yref_e; ia.xit = h->xit; ia.uit = h->uit;
    ia.W = static_cast<const real*>(h->W); ia.fac = static_cast<real*>(h->fac);
    ia.u0 = h->u0; ia.cost = h->cost; ia.status = h->status; ia.iters = h->iters; ia.rounds = h->rounds; ia.act = h->act;
    ia.timeline = h->timeline;
    if (h->reset_failed) ia.fail_streak = h->fail_streak;
    if (h->variant == 2) {
        // screening: warm-started active-set rounds in a Riccati kernel; whatever does not settle goes to the dense kernel.
        // With the warm start off there is nothing to screen: the dense kernel takes every OCP from its cold IPM.
        fill_screen_args(h->cfg, ia);
        const bool screen = ia.warm_rounds > 0;
        CU_TRY(cudaMemsetAsync(h->hard + B, 0, 2 * sizeof(int), S(stream)));
        if (screen) {
            // unsettled-after-screen_rounds counters of this and of the previous solve (ping-pong, no device copy)
            h->parity ^= 1;
            ia.unsettled_cur = h->hard + B + 2 + h->parity; ia.unsettled_prev = h->hard + B + 2 + (h->parity ^ 1);
            CU_TRY(cudaMemsetAsync(ia.unsettled_cur, 0, sizeof(int), S(stream)));
            ia.hard_list = h->hard; ia.hard_count = h->hard + B;
            const size_t smem_s = (size_t)IPM_WARPS * ia.smem_per_warp * sizeof(real);
            qmpc_ipm_kernel<real, IPM_WARPS><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem_s, S(stream)>>>(ia);
            LAUNCH_CHECK();
        }
        if (e2) {
            cudaEvent_t em = nullptr;
            CU_TRY(cudaEventCreate(&em));
            h->ev_mid.push_back(em);
            CU_TRY(cudaEventRecord(em, S(stream)));
        }
        DenseArgs<real> dn;
        dn.b = ia;
        dn.hard_list = screen ? h->hard : nullptr; dn.hard_count = screen ? h->hard + B : nullptr;
        dn.next_item = h->hard + B + 1;
        if constexpr (sizeof(real) == 8)
            qmpc_dense_kernel<real><<<h->dense_grid, DN_THREADS, dense_layout(N).total * sizeof(real), S(stream)>>>(dn);
    } else {
        const size_t smem = (size_t)IPM_WARPS * ia.smem_per_warp * sizeof(real);
        qmpc_ipm_kernel<real, IPM_WARPS><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem, S(stream)>>>(ia);
    }
    LAUNCH_CHECK();
    if (e2) CU_TRY(cudaEventRecord(e2, S(stream)));
    h->solved = true;
    return QMPC_OK;
}

// the handle's configuration with the weights of its last solve: the sensitivities differentiate that solve, whatever
// qmpc_set_weights has set for the next one
static qmpc_config solved_cfg(const qmpc_solver* h)
{
    qmpc_config c = h->cfg;
    std::memcpy(c.w_diag, h->w_solved, sizeof(c.w_diag));
    std::memcpy(c.we_diag, h->we_solved, sizeof(c.we_diag));
    return c;
}

static int sens_impl(qmpc_solver* h, int n_stages, double* sens_x, double* sens_u, void* stream)
{
    typedef double real;
    const int B = h->cfg.batch;
    SensArgs<real> sa;
    fill_sens_args(solved_cfg(h), n_stages, sa);
    sa.b.x0 = nullptr; sa.b.yref = nullptr; sa.b.yref_e = h->yref_e; sa.b.xit = h->xit; sa.b.uit = nullptr;
    sa.b.W = static_cast<const real*>(h->W); sa.b.fac = static_cast<real*>(h->fac); sa.b.act = h->act;
    sa.sens_x = sens_x; sa.sens_u = sens_u;
    const size_t smem = (size_t)IPM_WARPS * sa.b.smem_per_warp * sizeof(real);
    qmpc_sens_kernel<real, IPM_WARPS><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem, S(stream)>>>(sa);
    LAUNCH_CHECK();
    return QMPC_OK;
}

// weights: qmpc_eval_adjoint_weights (w_bar / we_bar, the kernel's WGT instantiation); otherwise qmpc_eval_adjoint
static int adjoint_impl(qmpc_solver* h, const double* x_bar, const double* u_bar, double* x0_bar, double* yref_bar,
                        double* yref_e_bar, bool weights, double* w_bar, double* we_bar, void* stream)
{
    typedef double real;
    const int B = h->cfg.batch;
    AdjArgs<real> aa;
    fill_sens_base(solved_cfg(h), aa.b);
    aa.b.x0 = nullptr; aa.b.yref = nullptr; aa.b.yref_e = h->yref_e; aa.b.xit = h->xit; aa.b.uit = nullptr;
    aa.b.W = static_cast<const real*>(h->W); aa.b.fac = static_cast<real*>(h->fac); aa.b.act = h->act;
    aa.x_bar = x_bar; aa.u_bar = u_bar; aa.x0_bar = x0_bar; aa.yref_bar = yref_bar; aa.yref_e_bar = yref_e_bar;
    aa.x = h->xit; aa.u = h->uit; aa.yref = h->yref; aa.yref_e = h->yref_e; aa.w_bar = w_bar; aa.we_bar = we_bar;
    const size_t smem = (size_t)IPM_WARPS * aa.b.smem_per_warp * sizeof(real);
    if (weights)
        qmpc_adjoint_kernel<real, IPM_WARPS, true><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem, S(stream)>>>(aa);
    else
        qmpc_adjoint_kernel<real, IPM_WARPS><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem, S(stream)>>>(aa);
    LAUNCH_CHECK();
    return QMPC_OK;
}

static int jvp_impl(qmpc_solver* h, int n_dir, const double* dx0, const double* dyref, const double* dyref_e,
                    const double* dw, const double* dwe, double* dx, double* du, void* stream)
{
    typedef double real;
    const int B = h->cfg.batch;
    JvpArgs<real> ja;
    fill_sens_base(solved_cfg(h), ja.b);
    ja.b.x0 = nullptr; ja.b.yref = nullptr; ja.b.yref_e = h->yref_e; ja.b.xit = h->xit; ja.b.uit = nullptr;
    ja.b.W = static_cast<const real*>(h->W); ja.b.fac = static_cast<real*>(h->fac); ja.b.act = h->act;
    ja.K = n_dir; ja.dx0 = dx0; ja.dyref = dyref; ja.dyref_e = dyref_e; ja.dw = dw; ja.dwe = dwe; ja.dx = dx; ja.du = du;
    ja.x = h->xit; ja.u = h->uit; ja.yref = h->yref; ja.yref_e = h->yref_e;
    const size_t smem = (size_t)IPM_WARPS * ja.b.smem_per_warp * sizeof(real);
    qmpc_jvp_kernel<real, IPM_WARPS><<<cdiv(B, IPM_WARPS), IPM_WARPS * 32, smem, S(stream)>>>(ja);
    LAUNCH_CHECK();
    return QMPC_OK;
}

extern "C" {

int qmpc_solve(qmpc_handle_t h, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return h->cfg.precision == 64 ? solve_impl<double>(h, stream) : solve_impl<float>(h, stream);
}

int qmpc_eval_sens_x0(qmpc_handle_t h, int n_stages, double* sens_x, double* sens_u, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (n_stages < 1 || n_stages > h->cfg.n_nodes) return fail(QMPC_ERR_ARG, "n_stages must be in [1, n_nodes]");
    if (!sens_u) return fail(QMPC_ERR_ARG, "sens_u is NULL");
    // fp32 tiles and an fp32 Riccati recursion without the solve's fp64 refinement: up to 1.4e-3 relative on a B200 (DESIGN §4)
    if (h->cfg.precision != 64) return fail(QMPC_ERR_ARG, "sensitivities need an fp64 handle (precision 64)");
    if (!h->solved) return fail(QMPC_ERR_ARG, "no solve on this handle yet: the sensitivities need its stage tiles");
    return sens_impl(h, n_stages, sens_x, sens_u, stream);
}

int qmpc_eval_adjoint(qmpc_handle_t h, const double* x_bar, const double* u_bar, double* x0_bar, double* yref_bar,
                      double* yref_e_bar, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (h->cfg.precision != 64) return fail(QMPC_ERR_ARG, "sensitivities need an fp64 handle (precision 64)");
    if (!h->solved) return fail(QMPC_ERR_ARG, "no solve on this handle yet: the sensitivities need its stage tiles");
    if (!x_bar && !u_bar) return fail(QMPC_ERR_ARG, "x_bar and u_bar are both NULL: nothing to differentiate");
    if (!x0_bar && !yref_bar && !yref_e_bar) return fail(QMPC_ERR_ARG, "x0_bar, yref_bar and yref_e_bar are all NULL");
    return adjoint_impl(h, x_bar, u_bar, x0_bar, yref_bar, yref_e_bar, false, nullptr, nullptr, stream);
}

int qmpc_eval_adjoint_weights(qmpc_handle_t h, const double* x_bar, const double* u_bar, double* x0_bar,
                              double* yref_bar, double* yref_e_bar, double* w_bar, double* we_bar, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (h->cfg.precision != 64) return fail(QMPC_ERR_ARG, "sensitivities need an fp64 handle (precision 64)");
    if (!h->solved) return fail(QMPC_ERR_ARG, "no solve on this handle yet: the sensitivities need its stage tiles");
    if (!x_bar && !u_bar) return fail(QMPC_ERR_ARG, "x_bar and u_bar are both NULL: nothing to differentiate");
    if (!x0_bar && !yref_bar && !yref_e_bar && !w_bar && !we_bar)
        return fail(QMPC_ERR_ARG, "x0_bar, yref_bar, yref_e_bar, w_bar and we_bar are all NULL");
    return adjoint_impl(h, x_bar, u_bar, x0_bar, yref_bar, yref_e_bar, true, w_bar, we_bar, stream);
}

int qmpc_eval_jvp(qmpc_handle_t h, int n_dir, const double* dx0, const double* dyref, const double* dyref_e,
                  const double* dw, const double* dwe, double* dx, double* du, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (h->cfg.precision != 64) return fail(QMPC_ERR_ARG, "sensitivities need an fp64 handle (precision 64)");
    if (!h->solved) return fail(QMPC_ERR_ARG, "no solve on this handle yet: the sensitivities need its stage tiles");
    if (n_dir < 1) return fail(QMPC_ERR_ARG, "n_dir must be >= 1");
    if (!dx0 && !dyref && !dyref_e && !dw && !dwe)
        return fail(QMPC_ERR_ARG, "dx0, dyref, dyref_e, dw and dwe are all NULL: nothing to differentiate");
    if (!du) return fail(QMPC_ERR_ARG, "du is NULL");
    return jvp_impl(h, n_dir, dx0, dyref, dyref_e, dw, dwe, dx, du, stream);
}

int qmpc_get_sens_epoch(qmpc_handle_t h, long long* epoch)
{
    if (!h || !epoch) return fail(QMPC_ERR_ARG, "null argument");
    *epoch = h->epoch;
    return QMPC_OK;
}

int qmpc_get_u0(qmpc_handle_t h, double* u0, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(u0, h->u0, (size_t)h->cfg.batch * NU * 8, stream);
}
int qmpc_get_x(qmpc_handle_t h, double* x, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(x, h->xit, (size_t)h->cfg.batch * (h->cfg.n_nodes + 1) * NX * 8, stream);
}
int qmpc_get_u(qmpc_handle_t h, double* u, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(u, h->uit, (size_t)h->cfg.batch * h->cfg.n_nodes * NU * 8, stream);
}
int qmpc_get_cost(qmpc_handle_t h, double* cost, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(cost, h->cost, (size_t)h->cfg.batch * 8, stream);
}
int qmpc_get_status(qmpc_handle_t h, int* status, int* iters, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    if (status) { int rc = copy_dd(status, h->status, (size_t)h->cfg.batch * 4, stream); if (rc) return rc; }
    if (iters) { int rc = copy_dd(iters, h->iters, (size_t)h->cfg.batch * 4, stream); if (rc) return rc; }
    return QMPC_OK;
}
int qmpc_get_fail_streak(qmpc_handle_t h, int* streak, void* stream)
{
    if (!h || !streak) return fail(QMPC_ERR_ARG, "null argument");
    return copy_dd(streak, h->fail_streak, (size_t)h->cfg.batch * 4, stream);
}
int qmpc_get_refine_rounds(qmpc_handle_t h, int* rounds, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(rounds, h->rounds, (size_t)h->cfg.batch * 4, stream);
}
int qmpc_get_hard_count(qmpc_handle_t h, int* count_host, void* stream)
{
    if (!h || !count_host) return fail(QMPC_ERR_ARG, "null argument");
    *count_host = 0;
    if (!h->hard) return QMPC_OK;
    CU_TRY(cudaMemcpyAsync(count_host, h->hard + h->cfg.batch, sizeof(int), cudaMemcpyDeviceToHost, S(stream)));
    CU_TRY(cudaStreamSynchronize(S(stream)));
    return QMPC_OK;
}
int qmpc_get_active_set(qmpc_handle_t h, unsigned char* act, void* stream)
{
    if (!h || !act) return fail(QMPC_ERR_ARG, "null argument");
    return copy_dd(act, h->act, (size_t)h->cfg.batch * h->cfg.n_nodes * NU, stream);
}
int qmpc_set_active_set(qmpc_handle_t h, const unsigned char* act, void* stream)
{
    if (!h || !act) return fail(QMPC_ERR_ARG, "null argument");
    ++h->epoch;
    return copy_dd(h->act, act, (size_t)h->cfg.batch * h->cfg.n_nodes * NU, stream);
}
int qmpc_reset_warm_start(qmpc_handle_t h, void* stream)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    ++h->epoch;
    CU_TRY(cudaMemsetAsync(h->act, 255, (size_t)h->cfg.batch * h->cfg.n_nodes * NU, S(stream)));
    return QMPC_OK;
}
int qmpc_iters_total(qmpc_handle_t h, long long* total, void* stream)
{
    if (!h || !total) return fail(QMPC_ERR_ARG, "null argument");
    std::vector<int> it(h->cfg.batch);
    CU_TRY(cudaMemcpyAsync(it.data(), h->iters, it.size() * 4, cudaMemcpyDeviceToHost, S(stream)));
    CU_TRY(cudaStreamSynchronize(S(stream)));
    long long s = 0;
    for (int v : it) s += v;
    *total = s;
    return QMPC_OK;
}

// ------------------------------------------------------------------------------------------ helpers

static void model_from_quad(const double* quad, ModelParams<double>& mp)
{
    qmpc_config c;
    std::memset(&c, 0, sizeof(c));
    std::memcpy(c.quad, quad, sizeof(c.quad));
    fill_model(c, mp);
    mp.M = 0;
}

int qmpc_predict_nominal(const double* quad, int B, const double* x, const double* u, double dt, int body_frame,
                         double* x_next, void* stream)
{
    if (!quad || !x || !u || !x_next || B < 1) return fail(QMPC_ERR_ARG, "bad argument");
    ModelParams<double> mp;
    model_from_quad(quad, mp);
    predict_nominal_kernel<<<cdiv(B, 128), 128, 0, S(stream)>>>(mp, B, x, u, dt, body_frame, x_next);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qmpc_compute_a_drag(int B, const double* x_now, const double* x_pred, double dt, double* v_body, double* a_drag,
                        void* stream)
{
    if (!x_now || !x_pred || !v_body || !a_drag || B < 1) return fail(QMPC_ERR_ARG, "bad argument");
    compute_a_drag_kernel<<<cdiv(B, 128), 128, 0, S(stream)>>>(B, x_now, x_pred, dt, v_body, a_drag);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qmpc_reference_chunk(int B, int K, const double* traj, int idx, int N, int skip, double* chunk, void* stream)
{
    if (!traj || !chunk || B < 1 || K < 1 || N < 1 || skip < 1 || idx < 0) return fail(QMPC_ERR_ARG, "bad argument");
    reference_chunk_kernel<<<cdiv((long long)B * N * NX, 256), 256, 0, S(stream)>>>(B, K, traj, idx, N, skip, chunk);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qmpc_reference_generate(int kind, int B, const double* params, int K, int idx, int N, int skip, double dt, double* chunk,
                            void* stream)
{
    if (!params || !chunk || B < 1 || K < 1 || N < 1 || skip < 1 || idx < 0 || kind < 0 || kind > 2 || !(dt > 0))
        return fail(QMPC_ERR_ARG, "bad argument");
    reference_generate_kernel<<<cdiv((long long)B * N, 128), 128, 0, S(stream)>>>(kind, B, params, K, idx, N, skip, dt, chunk);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qmpc_plant_period(const double* quad, const double* plant, int B, double* x, const double* u, double sim_dt,
                      int n_sub, void* stream)
{
    if (!quad || !plant || !x || !u || B < 1 || n_sub < 0) return fail(QMPC_ERR_ARG, "bad argument");
    ModelParams<double> mp;
    model_from_quad(quad, mp);
    PlantParams pp;
    pp.aero = plant[0]; pp.rotor[0] = plant[1]; pp.rotor[1] = plant[2]; pp.rotor[2] = plant[3]; pp.mass = quad[0];
    plant_period_kernel<<<cdiv(B, 128), 128, 0, S(stream)>>>(mp, pp, B, x, u, sim_dt, n_sub);
    LAUNCH_CHECK();
    return QMPC_OK;
}

// ---------------------------------------------------------------------------------------------- RGP

int qrgp_destroy(qrgp_handle_t g);

int qrgp_create(int batch, int n_basis, const double* X, const double* theta, const double* Kx, const double* Kx_inv,
                int device, qrgp_handle_t* out)
{
    if (!X || !theta || !Kx || !Kx_inv || !out) return fail(QMPC_ERR_ARG, "null argument");
    if (batch < 1 || n_basis < 1 || n_basis > 32 * RGP_MAXT) return fail(QMPC_ERR_ARG, "batch/n_basis out of range");
    CU_TRY(cudaSetDevice(device));
    std::unique_ptr<qrgp_model, int (*)(qrgp_handle_t)> guard(new qrgp_model(), qrgp_destroy);
    qrgp_model* g = guard.get();
    g->B = batch; g->M = n_basis; g->device = device;
    CU_TRY(cudaDeviceGetAttribute(&g->sms, cudaDevAttrMultiProcessorCount, device));
    const size_t B = batch, M = n_basis;
#define ALLOC(p, n) CU_TRY(cudaMalloc(reinterpret_cast<void**>(&(p)), (n)))
    ALLOC(g->X, 3 * M * 8); ALLOC(g->theta, 9 * 8); ALLOC(g->Kx, 3 * M * M * 8); ALLOC(g->Kx_inv, 3 * M * M * 8);
    ALLOC(g->mu, B * 3 * M * 8); ALLOC(g->C, B * 3 * M * M * 8); ALLOC(g->alpha, B * 3 * M * 8);
    ALLOC(g->xt, B * 3 * 8); ALLOC(g->yt, B * 3 * 8);
    if (batch == 1) {
        // shared-swarm mode: per-CTA partial sums of the information-form accumulate (no atomics: fixed summation order)
        const size_t per_warp = (size_t)(M * M + 3 * M) * 8;
        int warps = int((200 * 1024) / per_warp);
        g->acc_warps = warps > 8 ? 8 : warps;
        g->part_ctas = g->sms;
        if (g->acc_warps >= 1) {
            ALLOC(g->part, (size_t)3 * g->part_ctas * (M * M + M) * 8);
            const int smem = (int)(per_warp * g->acc_warps);
#define SHARED_ATTR(W) case W: CU_TRY(cudaFuncSetAttribute(qrgp_shared_accumulate_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); break;
            switch (g->acc_warps) { SHARED_ATTR(1) SHARED_ATTR(2) SHARED_ATTR(3) SHARED_ATTR(4) SHARED_ATTR(5) SHARED_ATTR(6) SHARED_ATTR(7) SHARED_ATTR(8) }
#undef SHARED_ATTR
        }
        const size_t smem_apply = (size_t)M * (2 * M + 1) * 8;
        if (smem_apply <= 220 * 1024)
            CU_TRY(cudaFuncSetAttribute(qrgp_shared_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_apply));
    }
#undef ALLOC
    CU_TRY(cudaMemcpy(g->X, X, 3 * M * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->theta, theta, 9 * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->Kx, Kx, 3 * M * M * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->Kx_inv, Kx_inv, 3 * M * M * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(g->mu, 0, B * 3 * M * 8));
    CU_TRY(cudaMemset(g->alpha, 0, B * 3 * M * 8));
    qrgp_fill_C_kernel<<<cdiv((long long)B * 3 * M * M, 256), 256>>>((long long)B, 3 * (int)M * (int)M, g->Kx, g->C);   // C0 = K_x for every vehicle (RGP.py:144)
    LAUNCH_CHECK();
    CU_TRY(cudaDeviceSynchronize());
    *out = guard.release();
    return QMPC_OK;
}

int qrgp_destroy(qrgp_handle_t g)
{
    if (!g) return QMPC_OK;
    cudaSetDevice(g->device);
    void* ps[] = {g->X, g->theta, g->Kx, g->Kx_inv, g->mu, g->C, g->alpha, g->xt, g->yt, g->part};
    for (void* p : ps) if (p) cudaFree(p);
    delete g;
    return QMPC_OK;
}

static int regress_launch(qrgp_model* g, const double* xt, const double* yt, void* stream)
{
    RgpArgs a;
    a.B = g->B; a.M = g->M; a.X = g->X; a.theta = g->theta; a.Kx_inv = g->Kx_inv; a.mu = g->mu; a.C = g->C;
    a.alpha = g->alpha; a.xt = xt; a.yt = yt;
    if (g->M % 2 == 0 && g->M <= RGP_TMA_MAXM) {
        // covariance staged through shared memory by TMA bulk copies; fewer warps per block as the per-model block grows
        const size_t per_warp = (size_t)rgp_tma_reals(g->M) * 8;
        const long long models = (long long)g->B * 3;
        if (per_warp * 8 <= 48 * 1024) {
            qrgp_regress_tma_kernel<8><<<cdiv(models, 8), 8 * 32, per_warp * 8, S(stream)>>>(a);
        } else if (per_warp * 2 <= 48 * 1024) {
            qrgp_regress_tma_kernel<2><<<cdiv(models, 2), 2 * 32, per_warp * 2, S(stream)>>>(a);
        } else {
            qrgp_regress_tma_kernel<1><<<models, 32, per_warp, S(stream)>>>(a);
        }
    } else {
        const size_t smem = (size_t)RGP_WARPS * 3 * g->M * 8;
        qrgp_regress_kernel<RGP_WARPS><<<cdiv((long long)g->B * 3, RGP_WARPS), RGP_WARPS * 32, smem, S(stream)>>>(a);
    }
    LAUNCH_CHECK();
    g->pushed = true;
    return QMPC_OK;
}

int qrgp_regress(qrgp_handle_t g, const double* xt, const double* yt, void* stream)
{
    if (!g || !xt || !yt) return fail(QMPC_ERR_ARG, "null argument");
    return regress_launch(g, xt, yt, stream);
}

int qrgp_regress_from_states(qrgp_handle_t g, const double* x_now, const double* x_pred_prev, double dt,
                             double* v_body, double* a_drag, void* stream)
{
    if (!g || !x_now || !x_pred_prev) return fail(QMPC_ERR_ARG, "null argument");
    compute_a_drag_kernel<<<cdiv(g->B, 128), 128, 0, S(stream)>>>(g->B, x_now, x_pred_prev, dt, g->xt, g->yt);
    LAUNCH_CHECK();
    if (v_body) { int rc = copy_dd(v_body, g->xt, (size_t)g->B * 3 * 8, stream); if (rc) return rc; }
    if (a_drag) { int rc = copy_dd(a_drag, g->yt, (size_t)g->B * 3 * 8, stream); if (rc) return rc; }
    return regress_launch(g, g->xt, g->yt, stream);
}

int qrgp_get_mu(qrgp_handle_t g, double* mu, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(mu, g->mu, (size_t)g->B * 3 * g->M * 8, stream);
}
int qrgp_get_C(qrgp_handle_t g, double* C, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(C, g->C, (size_t)g->B * 3 * g->M * g->M * 8, stream);
}
int qrgp_get_alpha(qrgp_handle_t g, double* alpha, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    return copy_dd(alpha, g->alpha, (size_t)g->B * 3 * g->M * 8, stream);
}
int qrgp_set_state(qrgp_handle_t g, const double* mu, const double* C, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    if (mu) {
        int rc = copy_dd(g->mu, mu, (size_t)g->B * 3 * g->M * 8, stream);
        if (rc) return rc;
        qrgp_alpha_kernel<<<cdiv((long long)g->B * 3 * g->M, 128), 128, 0, S(stream)>>>(g->B, g->M, g->Kx_inv, g->mu, g->alpha);
        LAUNCH_CHECK();
    }
    g->pushed = false;      // like the reference, a loaded/assigned model reaches the solver with the next regress
    if (C) return copy_dd(g->C, C, (size_t)g->B * 3 * g->M * g->M * 8, stream);
    return QMPC_OK;
}
const double* qrgp_Kx_inv_device(qrgp_handle_t g) { return g ? g->Kx_inv : nullptr; }
const double* qrgp_mu_device(qrgp_handle_t g) { return g ? g->mu : nullptr; }

static int predict_launch(qrgp_model* g, int m, const double* xs, const double* mu, const double* C, double* mean,
                          double* var, void* stream)
{
    RgpPredArgs a;
    a.B = g->B; a.M = g->M; a.m = m; a.X = g->X; a.theta = g->theta; a.Kx_inv = g->Kx_inv; a.mu = mu; a.C = C;
    a.xs = xs; a.mean = mean; a.var = var;
    const size_t smem = (size_t)RGP_WARPS * 2 * g->M * 8;
    qrgp_predict_kernel<RGP_WARPS><<<cdiv((long long)g->B * 3, RGP_WARPS), RGP_WARPS * 32, smem, S(stream)>>>(a);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qrgp_predict(qrgp_handle_t g, int m, const double* xs, double* mean, double* var, void* stream)
{
    if (!g || !xs || !mean || m < 1) return fail(QMPC_ERR_ARG, "bad argument");
    return predict_launch(g, m, xs, g->mu, g->C, mean, var, stream);
}

int qrgp_predict_cov(qrgp_handle_t g, int m, const double* xs, double* Jt, double* cov, void* stream)
{
    if (!g || !xs || !Jt || !cov || m < 1) return fail(QMPC_ERR_ARG, "bad argument");
    RgpCovArgs a;
    a.B = g->B; a.M = g->M; a.m = m; a.X = g->X; a.theta = g->theta; a.Kx_inv = g->Kx_inv; a.C = g->C; a.xs = xs; a.Jt = Jt; a.cov = cov;
    const size_t smem = (size_t)RGP_WARPS * g->M * 8;
    qrgp_predict_cov_kernel<RGP_WARPS><<<cdiv((long long)g->B * 3, RGP_WARPS), RGP_WARPS * 32, smem, S(stream)>>>(a);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qrgp_predict_using_y(qrgp_handle_t g, int m, const double* xs, const double* y, double* mean, void* stream)
{
    if (!g || !xs || !y || !mean || m < 1) return fail(QMPC_ERR_ARG, "bad argument");
    return predict_launch(g, m, xs, y, nullptr, mean, nullptr, stream);
}

int qrgp_shared_accumulate(qrgp_handle_t g, int B, const double* xt, const double* yt, double* info, void* stream)
{
    if (!g || !xt || !yt || !info || B < 1) return fail(QMPC_ERR_ARG, "bad argument");
    if (g->B != 1 || !g->part) return fail(QMPC_ERR_ARG, "shared model handles must be created with batch == 1 (n_basis small enough for the accumulate tile)");
    const int M = g->M, warps = g->acc_warps;
    const size_t per_warp = (size_t)(M * M + 3 * M) * 8;
    RgpSharedArgs a;
    a.B = B; a.M = M; a.X = g->X; a.theta = g->theta; a.Kx_inv = g->Kx_inv; a.xt = xt; a.yt = yt; a.part = g->part;
    int blocks = cdiv(B, warps * 8);
    blocks = blocks > g->part_ctas ? g->part_ctas : blocks;
    dim3 grid(blocks, 3);
    const size_t smem = per_warp * warps;
#define SHARED_LAUNCH(W) case W: qrgp_shared_accumulate_kernel<W><<<grid, W * 32, smem, S(stream)>>>(a); break;
    switch (warps) {
        SHARED_LAUNCH(1) SHARED_LAUNCH(2) SHARED_LAUNCH(3) SHARED_LAUNCH(4)
        SHARED_LAUNCH(5) SHARED_LAUNCH(6) SHARED_LAUNCH(7) SHARED_LAUNCH(8)
    }
#undef SHARED_LAUNCH
    LAUNCH_CHECK();
    // second stage: fixed-order sum of the per-CTA partials (results are bit-reproducible run to run)
    qrgp_shared_reduce_kernel<<<dim3(cdiv(M * M + M, 256), 3), 256, 0, S(stream)>>>(M * M + M, blocks, g->part_ctas, g->part, info);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qrgp_shared_apply(qrgp_handle_t g, const double* info, void* stream)
{
    if (!g || !info) return fail(QMPC_ERR_ARG, "null argument");
    if (g->B != 1) return fail(QMPC_ERR_ARG, "shared model handles must be created with batch == 1");
    const int M = g->M;
    const size_t smem = (size_t)M * (2 * M + 1) * 8;
    if (smem > 220 * 1024) return fail(QMPC_ERR_ARG, "n_basis too large for the shared apply tile");
    qrgp_shared_apply_kernel<<<3, 256, smem, S(stream)>>>(M, info, g->mu, g->C, g->Kx_inv, g->alpha);
    LAUNCH_CHECK();
    g->pushed = true;
    return QMPC_OK;
}

// --------------------------------------------------------------------------------------- fused step

int qmpc_step(qmpc_handle_t h, qrgp_handle_t g, const double* x_now, const double* x_ref, double* x_pred_prev,
              int first_step, double* u0_out, void* stream)
{
    return qmpc_step_dt(h, g, x_now, x_ref, x_pred_prev, first_step, u0_out, 0.0, stream);
}

int qmpc_step_dt(qmpc_handle_t h, qrgp_handle_t g, const double* x_now, const double* x_ref, double* x_pred_prev,
                 int first_step, double* u0_out, double odometry_dt, void* stream)
{
    if (!h || !x_now || !x_ref || !x_pred_prev) return fail(QMPC_ERR_ARG, "null argument");
    const double pred_dt = odometry_dt > 0 ? odometry_dt : h->dt;
    const int B = h->cfg.batch, N = h->cfg.n_nodes;
    if (g && (g->M != h->cfg.n_basis || (g->B != B && g->B != 1)))
        return fail(QMPC_ERR_ARG, "RGP handle does not match the solver (n_basis / batch)");
    set_reference_kernel<<<cdiv((long long)B * N * NY, 256), 256, 0, S(stream)>>>(B, N, x_ref, nullptr, 0.16, h->yref, h->yref_e);
    LAUNCH_CHECK();
    h->x0_src = x_now;
    const double* bound_alpha = h->alpha_src;
    const int bound_stride = h->alpha_stride;
    // the reference's solver parameters are whatever was last pushed: zeros (or qmpc_set_params/alpha) until the first
    // regress of this model (quad_opt.py:101,402-404)
    if (g && g->pushed) { h->alpha_src = g->alpha; h->alpha_stride = g->B == 1 ? 0 : 3 * g->M; }
    int rc = qmpc_solve(h, stream);
    h->x0_src = h->x0;
    h->alpha_src = bound_alpha; h->alpha_stride = bound_stride;
    if (rc) return rc;
    const bool per_vehicle = g && g->B == B;
    double* xt = per_vehicle ? g->xt : h->xt;
    double* yt = per_vehicle ? g->yt : h->yt;
    post_solve_kernel<<<cdiv(B, 128), 128, 0, S(stream)>>>(h->mp64, B, pred_dt, first_step, x_now, h->u0, x_pred_prev,
                                                           g ? xt : nullptr, g ? yt : nullptr);
    LAUNCH_CHECK();
    if (per_vehicle) { rc = regress_launch(g, xt, yt, stream); if (rc) return rc; }
    if (u0_out) return copy_dd(u0_out, h->u0, (size_t)B * NU * 8, stream);
    return QMPC_OK;
}

/* One closed-loop control step entirely on `stream` (execute_trajectory.py:196-277 incl. the plant period):
 * reference chunk at `idx` of traj [B][K][13] -> qmpc_step -> plant advance of x [B][13] with u0. */
int qmpc_closed_loop_step(qmpc_handle_t h, qrgp_handle_t g, const double* traj, int K, int idx, double* x,
                          double* x_pred_prev, double* chunk, double* u0, const double* plant, double sim_dt, int n_sub,
                          void* stream)
{
    if (!h || !traj || !x || !x_pred_prev || !chunk || !u0 || !plant) return fail(QMPC_ERR_ARG, "null argument");
    const int B = h->cfg.batch, N = h->cfg.n_nodes;
    int rc = qmpc_reference_chunk(B, K, traj, idx, N, 1, chunk, stream);
    if (rc) return rc;
    rc = qmpc_step(h, g, x, chunk, x_pred_prev, idx == 0, u0, stream);
    if (rc) return rc;
    return qmpc_plant_period(h->cfg.quad, plant, B, x, u0, sim_dt, n_sub, stream);
}

// ------------------------------------------------------------------------------------------- RGP* learning

int qrgpl_destroy(qrgpl_handle_t g);

int qrgpl_create(int n_models, int n_basis, const double* X, const double* theta, int device, qrgpl_handle_t* out)
{
    if (!X || !theta || !out) return fail(QMPC_ERR_ARG, "null argument");
    if (n_models < 1 || n_basis < 1 || n_basis > 64) return fail(QMPC_ERR_ARG, "n_models / n_basis out of range (n_basis <= 64)");
    CU_TRY(cudaSetDevice(device));
    const size_t n = n_models, M = n_basis;
    // prior exactly as RGP.__init__: K_x = K(X,X) + sn^2 I, inverse by Gauss-Jordan with partial pivoting (host, once)
    std::vector<double> Kx(M * M), W(M * 2 * M);
    const double L = theta[0], sf = theta[1], sn = theta[2];
    for (size_t i = 0; i < M; ++i)
        for (size_t j = 0; j < M; ++j) {
            const double e = X[i] - X[j];
            const double k = sf * sf * std::exp(-0.5 * e * (1.0 / (L * L)) * e) + (i == j ? sn * sn : 0.0);
            Kx[i * M + j] = k; W[i * 2 * M + j] = k; W[i * 2 * M + M + j] = (i == j);
        }
    for (size_t c = 0; c < M; ++c) {
        size_t piv = c;
        for (size_t i = c + 1; i < M; ++i) if (std::fabs(W[i * 2 * M + c]) > std::fabs(W[piv * 2 * M + c])) piv = i;
        if (W[piv * 2 * M + c] == 0) return fail(QMPC_ERR_ARG, "K_x is singular");
        if (piv != c) for (size_t j = 0; j < 2 * M; ++j) std::swap(W[c * 2 * M + j], W[piv * 2 * M + j]);
        const double d = 1.0 / W[c * 2 * M + c];
        for (size_t j = 0; j < 2 * M; ++j) W[c * 2 * M + j] *= d;
        for (size_t i = 0; i < M; ++i) if (i != c) {
            const double f = W[i * 2 * M + c];
            if (f != 0) for (size_t j = 0; j < 2 * M; ++j) W[i * 2 * M + j] -= f * W[c * 2 * M + j];
        }
    }
    std::vector<double> Kxi(M * M);
    for (size_t i = 0; i < M; ++i) for (size_t j = 0; j < M; ++j) Kxi[i * M + j] = W[i * 2 * M + M + j];
    std::unique_ptr<qrgpl_model, int (*)(qrgpl_handle_t)> guard(new qrgpl_model(), qrgpl_destroy);     // released on every early return
    qrgpl_model* g = guard.get();
    g->n = n_models; g->M = n_basis; g->device = device;
#define ALLOC(p, nb) CU_TRY(cudaMalloc(reinterpret_cast<void**>(&(p)), (nb)))
    ALLOC(g->X, M * 8); ALLOC(g->mu_g, n * M * 8); ALLOC(g->C_g, n * M * M * 8); ALLOC(g->mu_eta, n * 3 * 8);
    ALLOC(g->C_eta, n * 9 * 8); ALLOC(g->C_g_eta, n * M * 3 * 8); ALLOC(g->Kx_inv, n * M * M * 8); ALLOC(g->status, n * 4);
#undef ALLOC
    CU_TRY(cudaMemcpy(g->X, X, M * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(g->mu_g, 0, n * M * 8)); CU_TRY(cudaMemset(g->C_g_eta, 0, n * M * 3 * 8)); CU_TRY(cudaMemset(g->status, 0, n * 4));
    std::vector<double> eta(n * 3), Ce(n * 9, 0.0);
    for (size_t m = 0; m < n; ++m) { for (int k = 0; k < 3; ++k) { eta[m * 3 + k] = theta[k]; Ce[m * 9 + k * 4] = 1.0; } }
    CU_TRY(cudaMemcpy(g->mu_eta, eta.data(), n * 3 * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->C_eta, Ce.data(), n * 9 * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->C_g, Kx.data(), M * M * 8, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemcpy(g->Kx_inv, Kxi.data(), M * M * 8, cudaMemcpyHostToDevice));
    for (size_t m = 1; m < n; ++m) {
        CU_TRY(cudaMemcpyAsync(g->C_g + m * M * M, g->C_g, M * M * 8, cudaMemcpyDeviceToDevice, 0));
        CU_TRY(cudaMemcpyAsync(g->Kx_inv + m * M * M, g->Kx_inv, M * M * 8, cudaMemcpyDeviceToDevice, 0));
    }
    const int smem = rgp_learn_smem_doubles(n_basis) * 8;
    CU_TRY(cudaFuncSetAttribute(qrgp_learn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CU_TRY(cudaDeviceSynchronize());
    *out = guard.release();
    return QMPC_OK;
}

int qrgpl_destroy(qrgpl_handle_t g)
{
    if (!g) return QMPC_OK;
    cudaSetDevice(g->device);
    void* ps[] = {g->X, g->mu_g, g->C_g, g->mu_eta, g->C_eta, g->C_g_eta, g->Kx_inv, g->status};
    for (void* p : ps) if (p) cudaFree(p);
    delete g;
    return QMPC_OK;
}

int qrgpl_learn(qrgpl_handle_t g, const double* xt, const double* yt, double* mu_z, double* C_z, void* stream)
{
    if (!g || !xt || !yt) return fail(QMPC_ERR_ARG, "null argument");
    RgpLearnArgs a;
    a.n_models = g->n; a.M = g->M; a.X = g->X; a.mu_g = g->mu_g; a.C_g = g->C_g; a.mu_eta = g->mu_eta; a.C_eta = g->C_eta;
    a.C_g_eta = g->C_g_eta; a.Kx_inv = g->Kx_inv; a.mu_z = mu_z; a.C_z = C_z; a.xt = xt; a.yt = yt; a.status = g->status;
    qrgp_learn_kernel<<<g->n, 128, rgp_learn_smem_doubles(g->M) * 8, S(stream)>>>(a);
    LAUNCH_CHECK();
    return QMPC_OK;
}

int qrgpl_get_state(qrgpl_handle_t g, double* mu_g, double* C_g, double* mu_eta, double* C_eta, double* Kx_inv, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    const size_t n = g->n, M = g->M;
    int rc = 0;
    if (mu_g && !rc) rc = copy_dd(mu_g, g->mu_g, n * M * 8, stream);
    if (C_g && !rc) rc = copy_dd(C_g, g->C_g, n * M * M * 8, stream);
    if (mu_eta && !rc) rc = copy_dd(mu_eta, g->mu_eta, n * 3 * 8, stream);
    if (C_eta && !rc) rc = copy_dd(C_eta, g->C_eta, n * 9 * 8, stream);
    if (Kx_inv && !rc) rc = copy_dd(Kx_inv, g->Kx_inv, n * M * M * 8, stream);
    return rc;
}

int qrgpl_set_state(qrgpl_handle_t g, const double* mu_g, const double* C_g, const double* mu_eta, const double* C_eta,
                    const double* C_g_eta, const double* Kx_inv, void* stream)
{
    if (!g) return fail(QMPC_ERR_ARG, "null handle");
    const size_t n = g->n, M = g->M;
    int rc = 0;
    if (mu_g && !rc) rc = copy_dd(g->mu_g, mu_g, n * M * 8, stream);
    if (C_g && !rc) rc = copy_dd(g->C_g, C_g, n * M * M * 8, stream);
    if (mu_eta && !rc) rc = copy_dd(g->mu_eta, mu_eta, n * 3 * 8, stream);
    if (C_eta && !rc) rc = copy_dd(g->C_eta, C_eta, n * 9 * 8, stream);
    if (C_g_eta && !rc) rc = copy_dd(g->C_g_eta, C_g_eta, n * M * 3 * 8, stream);
    if (Kx_inv && !rc) rc = copy_dd(g->Kx_inv, Kx_inv, n * M * M * 8, stream);
    return rc;
}

int qrgpl_get_status(qrgpl_handle_t g, int* status, void* stream)
{
    if (!g || !status) return fail(QMPC_ERR_ARG, "null argument");
    return copy_dd(status, g->status, (size_t)g->n * 4, stream);
}

/* kernel timing for the roofline leg of bench.py: enable, run solves, then read (synchronises the device).
 * ms_lin / ms_ipm = summed device time of the linearize / ipm launches since enabling; count = solves timed. */
int qmpc_timing_enable(qmpc_handle_t h, int on)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->ev_mid) cudaEventDestroy(e);
    h->ev.clear(); h->ev_mid.clear();
    h->timing = on != 0;
    return QMPC_OK;
}
int qmpc_timeline_enable(qmpc_handle_t h, int on)
{
    if (!h) return fail(QMPC_ERR_ARG, "null handle");
    CU_TRY(cudaSetDevice(h->cfg.device));
    CU_TRY(cudaDeviceSynchronize());
    if (on && !h->timeline) {
        CU_TRY(cudaMalloc(reinterpret_cast<void**>(&h->timeline), (size_t)h->cfg.batch * 16));
        CU_TRY(cudaMemset(h->timeline, 0, (size_t)h->cfg.batch * 16));
    } else if (!on && h->timeline) {
        cudaFree(h->timeline);
        h->timeline = nullptr;
    }
    return QMPC_OK;
}
int qmpc_timeline_read(qmpc_handle_t h, long long* out)
{
    if (!h || !out) return fail(QMPC_ERR_ARG, "null argument");
    if (!h->timeline) return fail(QMPC_ERR_ARG, "timeline not enabled");
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(out, h->timeline, (size_t)h->cfg.batch * 16, cudaMemcpyDeviceToHost));
    return QMPC_OK;
}
int qmpc_timing_read_dense(qmpc_handle_t h, double* ms_dense)
{
    if (!h || !ms_dense) return fail(QMPC_ERR_ARG, "null argument");
    CU_TRY(cudaDeviceSynchronize());
    double d = 0;
    for (size_t i = 0; i < h->ev_mid.size() && 3 * i + 2 < h->ev.size(); ++i) {
        float t = 0;
        CU_TRY(cudaEventElapsedTime(&t, h->ev_mid[i], h->ev[3 * i + 2]));
        d += t;
    }
    *ms_dense = d;
    return QMPC_OK;
}
int qmpc_timing_read(qmpc_handle_t h, double* ms_lin, double* ms_ipm, int* count)
{
    if (!h || !ms_lin || !ms_ipm || !count) return fail(QMPC_ERR_ARG, "null argument");
    CU_TRY(cudaDeviceSynchronize());
    double a = 0, b = 0;
    for (size_t i = 0; i + 2 < h->ev.size(); i += 3) {
        float t1 = 0, t2 = 0;
        CU_TRY(cudaEventElapsedTime(&t1, h->ev[i], h->ev[i + 1]));
        CU_TRY(cudaEventElapsedTime(&t2, h->ev[i + 1], h->ev[i + 2]));
        a += t1; b += t2;
    }
    *ms_lin = a; *ms_ipm = b; *count = int(h->ev.size() / 3);
    return QMPC_OK;
}

/* register-resident FMA microbenchmark: measured non-tensor FMA peak of this GPU (TFLOP/s), precision 64 or 32 */
int qmpc_fma_peak(int precision, double* tflops, void* stream)
{
    if (!tflops || (precision != 64 && precision != 32)) return fail(QMPC_ERR_ARG, "bad argument");
    int dev = 0, sms = 0;
    CU_TRY(cudaGetDevice(&dev));
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 8, threads = 256, iters = 4096;
    struct Scratch {            // released on every return path
        double* sink = nullptr; cudaEvent_t e0 = nullptr, e1 = nullptr;
        ~Scratch() { if (e0) cudaEventDestroy(e0); if (e1) cudaEventDestroy(e1); if (sink) cudaFree(sink); }
    } sc;
    CU_TRY(cudaMalloc(&sc.sink, 8));
    CU_TRY(cudaEventCreate(&sc.e0)); CU_TRY(cudaEventCreate(&sc.e1));
    float best = 1e30f;
    for (int rep = 0; rep < 6; ++rep) {
        CU_TRY(cudaEventRecord(sc.e0, S(stream)));
        if (precision == 64) fma_peak_kernel<double><<<blocks, threads, 0, S(stream)>>>(iters, sc.sink);
        else fma_peak_kernel<float><<<blocks, threads, 0, S(stream)>>>(iters, sc.sink);
        LAUNCH_CHECK();
        CU_TRY(cudaEventRecord(sc.e1, S(stream)));
        CU_TRY(cudaEventSynchronize(sc.e1));
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, sc.e0, sc.e1));
        if (rep > 0 && ms < best) best = ms;
    }
    *tflops = 2.0 * 16.0 * iters * (double)blocks * threads / (best * 1e-3) / 1e12;
    return QMPC_OK;
}

/* residual buffers written by qmpc_step (v_body, a_drag of the last step), for the shared-swarm exchange */
const double* qmpc_residual_x_device(qmpc_handle_t h) { return h ? h->xt : nullptr; }
const double* qmpc_residual_y_device(qmpc_handle_t h) { return h ? h->yt : nullptr; }

}  // extern "C"
