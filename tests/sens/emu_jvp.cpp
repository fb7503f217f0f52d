// tests/sens/emu_jvp.cpp — TEST-ONLY.  qmpc_jvp_kernel (qmpc_eval_jvp) compiled for the host under the lane emulation of
// tests/emu (emu_cuda.h), run on the stage tiles and active set an emulated solve (tests/emu) returns.  Built by
// tests/sens/jvp_ref.py with the defines of the chosen tests/emu build flavour.
#define QMPC_EMU 1
#include "emu_cuda.h"
#include "../../mpc_quad_ros_b200/csrc/mpc_kernels.cuh"
#include "../../mpc_quad_ros_b200/csrc/host_params.h"

using namespace qmpc;

// qmpc_eval_jvp on the tiles and active set of an emulated fp64 solve, with that solve's solution x [B][N+1][13],
// u [B][N][4] and the reference yref [B][N][17], yref_e [B][13] it ran with.  n_dir directions per vehicle; the tangents
// and dx may be null.  The set-up of the costate offset is that of emu_adjoint_weights_f64.
extern "C" int emu_jvp_f64(const HostOcp* o, const double* Win, const unsigned char* act, int n_dir, const double* dx0,
                           const double* dyref, const double* dyref_e, const double* dw, const double* dwe,
                           const double* x, const double* u, const double* yref, const double* yref_e, double* dx,
                           double* du)
{
    typedef double real;
    const int B = o->batch, N = o->n_nodes;
    std::vector<real> W(((size_t)B * N + 1) * WT), fac((size_t)B * N * FAC);
    std::memcpy(W.data(), Win, (size_t)B * N * WT * sizeof(real));
    std::vector<double> xit((size_t)B * (N + 1) * NX, 0.0), yref_e0((size_t)B * NX, 0.0);
    std::vector<unsigned char> a(act, act + (size_t)B * N * NU);
    JvpArgs<real> ja;
    fill_sens_base(*o, ja.b);
    ja.b.x0 = nullptr; ja.b.yref = nullptr; ja.b.yref_e = yref_e0.data(); ja.b.xit = xit.data(); ja.b.uit = nullptr;
    ja.b.W = W.data(); ja.b.fac = fac.data(); ja.b.act = a.data();
    ja.K = n_dir; ja.dx0 = dx0; ja.dyref = dyref; ja.dyref_e = dyref_e; ja.dw = dw; ja.dwe = dwe; ja.dx = dx; ja.du = du;
    ja.x = x; ja.u = u; ja.yref = yref; ja.yref_e = yref_e;
    constexpr int WARPS = 4;
    emu::launch((B + WARPS - 1) / WARPS, WARPS * 32, (size_t)WARPS * ja.b.smem_per_warp * sizeof(real),
                [&]() { qmpc_jvp_kernel<real, WARPS>(ja); });
    return 0;
}
