"""TEST-ONLY: the two references of tests/test_adjoint_weights.py, built on first use next to their sources.

rti_adjoint_weights  -> tests/sens/rti_adjoint_weights.c: the formula on the oracle's linearisation and LQR routines
emu_adjoint_weights  -> tests/sens/emu_adjoint_weights.cpp: the product's qmpc_adjoint_kernel<.., true> under the lane
                        emulation of tests/emu"""
import ctypes as C
import os

import numpy as np

from emu import emu
from oracle import oracle as orc
from sens.sens_ref import _build, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIBS = {}
NX, NU = 13, 4


def _oracle_lib():
    if "oracle" not in _LIBS:
        src = os.path.join(_HERE, "rti_adjoint_weights.c")
        so = _build("librti_adjoint_weights.so",
                    lambda so: ["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-o", so, src, "-lm"],
                    [src, os.path.join(_ROOT, "oracle", "qmpc_oracle.c")])
        _LIBS["oracle"] = C.CDLL(so)
    return _LIBS["oracle"]


def _emu_lib(flavour):
    key = "emu_" + flavour
    if key not in _LIBS:
        defs, _ = emu.FLAVOURS[flavour]
        src = os.path.join(_HERE, "emu_adjoint_weights.cpp")
        emu_dir = os.path.join(_ROOT, "tests", "emu")
        csrc = os.path.join(_ROOT, "mpc_quad_ros_b200", "csrc")
        srcs = [src, os.path.join(emu_dir, "emu_cuda.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                             if f.endswith((".cuh", ".h"))]
        so = _build("libemu_adjoint_weights%s.so" % ("_" + flavour if flavour else ""),
                    lambda so: ["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", emu_dir] + defs +
                               ["-o", so, src], srcs)
        _LIBS[key] = C.CDLL(so)
    return _LIBS[key]


def rti_adjoint_weights(quad, dt, N, xit, uit, act, x, u, yref, yref_e, x_bar=None, u_bar=None, gp=None, alpha=None,
                        Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    """The gradients of <x_bar, x> + <u_bar, u> w.r.t. the cost weights Wd [17] and Wed [13] at the explicit active set
    act [4N]; x [N+1,13], u [N,4]: the step's solution, yref [N,17], yref_e [13] its reference; xit, uit: the PRE-solve
    iterate.  returns (w_bar [17], we_bar [13])"""
    assert xit.shape == (N + 1, NX) and uit.shape == (N, NU) and x.shape == (N + 1, NX) and u.shape == (N, NU)
    act = np.ascontiguousarray(act, dtype=np.uint8).reshape(N * NU)
    wb, web = np.empty(NX + NU), np.empty(NX)
    c = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    M = gp.M if gp is not None else 0
    args = [c(a) for a in (quad, alpha, Wd, Wed, xit, uit, x_bar, u_bar, x, u, yref, yref_e)]   # alive until the call returns
    quad, alpha, Wd, Wed, xit, uit, x_bar, u_bar, x, u, yref, yref_e = args
    ok = _oracle_lib().orc_rti_adjoint_weights(_p(quad), C.c_double(dt), N, M, _p(gp.X if gp else None),
                                               _p(gp.theta if gp else None), _p(alpha), _p(Wd), _p(Wed), _p(xit),
                                               _p(uit), _p(act), _p(x_bar), _p(u_bar), _p(x), _p(u), _p(yref),
                                               _p(yref_e), _p(wb), _p(web))
    assert ok == 1, "non-positive-definite factorisation in orc_rti_adjoint_weights"
    return wb, web


def emu_adjoint_weights(cfg, r, x, u, yref, yref_e, x_bar=None, u_bar=None, outputs=(True,) * 5, flavour=""):
    """qmpc_eval_adjoint_weights emulated on an fp64 emu.solve result `r`, its solution x [B,N+1,13], u [B,N,4] and the
    reference yref [B,N,17], yref_e [B,13] it ran with; outputs: which of (x0_bar, yref_bar, yref_e_bar, w_bar, we_bar)
    to ask for (the others come back None).  returns those five arrays ([B,13], [B,N,17], [B,13], [B,17], [B,13])"""
    B, N = cfg.batch, cfg.n_nodes
    W, act = np.ascontiguousarray(r["W"]), np.ascontiguousarray(r["act"], dtype=np.uint8)
    assert W.dtype == np.float64 and W.shape[-1] == emu.FLAVOURS[flavour][1]
    shapes = ((B, NX), (B, N, NX + NU), (B, NX), (B, NX + NU), (B, NX))
    out = [np.empty(s) if want else None for s, want in zip(shapes, outputs)]
    xb = None if x_bar is None else np.ascontiguousarray(x_bar, dtype=np.float64).reshape(B, N + 1, NX)
    ub = None if u_bar is None else np.ascontiguousarray(u_bar, dtype=np.float64).reshape(B, N, NU)
    sol = [np.ascontiguousarray(a, dtype=np.float64).reshape(s) for a, s in
           ((x, (B, N + 1, NX)), (u, (B, N, NU)), (yref, (B, N, NX + NU)), (yref_e, (B, NX)))]
    _emu_lib(flavour).emu_adjoint_weights_f64(C.byref(cfg), _p(W), _p(act), _p(xb), _p(ub), *(_p(a) for a in sol),
                                              *(_p(o) for o in out))
    return tuple(out)
