// tests/sens/emu_sens.cpp — TEST-ONLY.  qmpc_sens_kernel compiled for the host under the lane emulation of tests/emu
// (emu_cuda.h), run on the stage tiles and active set an emulated solve (tests/emu) returns.  Built by
// tests/sens/sens_ref.py with the defines of the chosen tests/emu build flavour.
#define QMPC_EMU 1
#include "emu_cuda.h"
#include "../../mpc_quad_ros_b200/csrc/mpc_kernels.cuh"
#include "../../mpc_quad_ros_b200/csrc/host_params.h"

using namespace qmpc;

// qmpc_eval_sens_x0 on the tiles Win [B][N][13][WR] and the active set act [B][4N] of an emulated fp64 solve (the library
// serves fp64 handles only)
template <typename real>
static int run_sens(const HostOcp* o, const real* Win, const unsigned char* act, int n_stages, double* sens_x, double* sens_u)
{
    const int B = o->batch, N = o->n_nodes;
    std::vector<real> W(((size_t)B * N + 1) * WT), fac((size_t)B * N * FAC);
    std::memcpy(W.data(), Win, (size_t)B * N * WT * sizeof(real));
    std::vector<double> xit((size_t)B * (N + 1) * NX, 0.0), yref_e((size_t)B * NX, 0.0);
    std::vector<unsigned char> a(act, act + (size_t)B * N * NU);
    SensArgs<real> sa;
    fill_sens_args(*o, n_stages, sa);
    sa.b.x0 = nullptr; sa.b.yref = nullptr; sa.b.yref_e = yref_e.data(); sa.b.xit = xit.data(); sa.b.uit = nullptr;
    sa.b.W = W.data(); sa.b.fac = fac.data(); sa.b.act = a.data();
    sa.sens_x = sens_x; sa.sens_u = sens_u;
    constexpr int WARPS = 4;
    emu::launch((B + WARPS - 1) / WARPS, WARPS * 32, (size_t)WARPS * sa.b.smem_per_warp * sizeof(real),
                [&]() { qmpc_sens_kernel<real, WARPS>(sa); });
    return 0;
}

extern "C" int emu_sens_f64(const HostOcp* o, const double* W, const unsigned char* act, int n_stages, double* sens_x, double* sens_u)
{
    return run_sens<double>(o, W, act, n_stages, sens_x, sens_u);
}
