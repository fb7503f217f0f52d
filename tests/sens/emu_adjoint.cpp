// tests/sens/emu_adjoint.cpp — TEST-ONLY.  qmpc_adjoint_kernel compiled for the host under the lane emulation of tests/emu
// (emu_cuda.h), run on the stage tiles and active set an emulated solve (tests/emu) returns.  Built by
// tests/sens/adjoint_ref.py with the defines of the chosen tests/emu build flavour.
#define QMPC_EMU 1
#include "emu_cuda.h"
#include "../../mpc_quad_ros_b200/csrc/mpc_kernels.cuh"
#include "../../mpc_quad_ros_b200/csrc/host_params.h"

using namespace qmpc;

// qmpc_eval_adjoint on the tiles and active set of an emulated fp64 solve; x_bar / u_bar and every output may be null
extern "C" int emu_adjoint_f64(const HostOcp* o, const double* Win, const unsigned char* act, const double* x_bar,
                               const double* u_bar, double* x0_bar, double* yref_bar, double* yref_e_bar)
{
    typedef double real;
    const int B = o->batch, N = o->n_nodes;
    std::vector<real> W(((size_t)B * N + 1) * WT), fac((size_t)B * N * FAC);
    std::memcpy(W.data(), Win, (size_t)B * N * WT * sizeof(real));
    std::vector<double> xit((size_t)B * (N + 1) * NX, 0.0), yref_e((size_t)B * NX, 0.0);
    std::vector<unsigned char> a(act, act + (size_t)B * N * NU);
    AdjArgs<real> aa;
    fill_sens_base(*o, aa.b);
    aa.b.x0 = nullptr; aa.b.yref = nullptr; aa.b.yref_e = yref_e.data(); aa.b.xit = xit.data(); aa.b.uit = nullptr;
    aa.b.W = W.data(); aa.b.fac = fac.data(); aa.b.act = a.data();
    aa.x_bar = x_bar; aa.u_bar = u_bar; aa.x0_bar = x0_bar; aa.yref_bar = yref_bar; aa.yref_e_bar = yref_e_bar;
    constexpr int WARPS = 4;
    emu::launch((B + WARPS - 1) / WARPS, WARPS * 32, (size_t)WARPS * aa.b.smem_per_warp * sizeof(real),
                [&]() { qmpc_adjoint_kernel<real, WARPS>(aa); });
    return 0;
}
