"""TEST-ONLY: the two references of tests/test_jvp.py, built on first use next to their sources.

rti_jvp  -> tests/sens/rti_jvp.c: the oracle's linearisation and LQR routines with the forward mode's linear costs
emu_jvp  -> tests/sens/emu_jvp.cpp: the product's qmpc_jvp_kernel under the lane emulation of tests/emu"""
import ctypes as C
import os

import numpy as np

from emu import emu
from oracle import oracle as orc
from sens.sens_ref import _build, _p

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIBS = {}
NX, NU, NY = 13, 4, 17


def _oracle_lib():
    if "oracle" not in _LIBS:
        src = os.path.join(_HERE, "rti_jvp.c")
        so = _build("librti_jvp.so",
                    lambda so: ["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-o", so, src, "-lm"],
                    [src, os.path.join(_ROOT, "oracle", "qmpc_oracle.c")])
        _LIBS["oracle"] = C.CDLL(so)
    return _LIBS["oracle"]


def _emu_lib(flavour):
    key = "emu_" + flavour
    if key not in _LIBS:
        defs, _ = emu.FLAVOURS[flavour]
        src = os.path.join(_HERE, "emu_jvp.cpp")
        emu_dir = os.path.join(_ROOT, "tests", "emu")
        csrc = os.path.join(_ROOT, "mpc_quad_ros_b200", "csrc")
        srcs = [src, os.path.join(emu_dir, "emu_cuda.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                             if f.endswith((".cuh", ".h"))]
        so = _build("libemu_jvp%s.so" % ("_" + flavour if flavour else ""),
                    lambda so: ["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", emu_dir] + defs +
                               ["-o", so, src], srcs)
        _LIBS[key] = C.CDLL(so)
    return _LIBS[key]


def rti_jvp(quad, dt, N, xit, uit, act, x, u, yref, yref_e, dx0=None, dyref=None, dyref_e=None, dw=None, dwe=None,
            gp=None, alpha=None, Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    """Forward mode of oracle.rti_step's result at the explicit active set act [4N] for the tangents dx0 [13],
    dyref [N,17], dyref_e [13], dw [17], dwe [13] (None = zero); x [N+1,13], u [N,4]: the step's solution, yref [N,17],
    yref_e [13] its reference; xit, uit: the PRE-solve iterate.  returns (dx [N+1,13], du [N,4])"""
    assert xit.shape == (N + 1, NX) and uit.shape == (N, NU) and x.shape == (N + 1, NX) and u.shape == (N, NU)
    act = np.ascontiguousarray(act, dtype=np.uint8).reshape(N * NU)
    dx, du = np.empty((N + 1, NX)), np.empty((N, NU))
    c = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    M = gp.M if gp is not None else 0
    args = [c(a) for a in (quad, alpha, Wd, Wed, xit, uit, x, u, yref, yref_e, dx0, dyref, dyref_e, dw, dwe)]
    quad, alpha, Wd, Wed, xit, uit, x, u, yref, yref_e, dx0, dyref, dyref_e, dw, dwe = args   # alive during the call
    ok = _oracle_lib().orc_rti_jvp(_p(quad), C.c_double(dt), N, M, _p(gp.X if gp else None),
                                   _p(gp.theta if gp else None), _p(alpha), _p(Wd), _p(Wed), _p(xit), _p(uit),
                                   _p(act), _p(x), _p(u), _p(yref), _p(yref_e), _p(dx0), _p(dyref), _p(dyref_e),
                                   _p(dw), _p(dwe), _p(dx), _p(du))
    assert ok == 1, "non-positive-definite factorisation in orc_rti_jvp"
    return dx, du


def emu_jvp(cfg, r, x, u, yref, yref_e, dx0=None, dyref=None, dyref_e=None, dw=None, dwe=None, n_dir=1, states=True,
            flavour=""):
    """qmpc_eval_jvp emulated on an fp64 emu.solve result `r`, its solution x [B,N+1,13], u [B,N,4] and the reference
    yref [B,N,17], yref_e [B,13] it ran with; tangents [B,K,13], [B,K,N,17], [B,K,13], [B,K,17], [B,K,13] or None.
    returns (dx [B,K,N+1,13] or None when states=False, du [B,K,N,4])"""
    B, N, K = cfg.batch, cfg.n_nodes, n_dir
    W, act = np.ascontiguousarray(r["W"]), np.ascontiguousarray(r["act"], dtype=np.uint8)
    assert W.dtype == np.float64 and W.shape[-1] == emu.FLAVOURS[flavour][1]
    tan = [None if t is None else np.ascontiguousarray(t, dtype=np.float64).reshape(s) for t, s in
           ((dx0, (B, K, NX)), (dyref, (B, K, N, NY)), (dyref_e, (B, K, NX)), (dw, (B, K, NY)), (dwe, (B, K, NX)))]
    sol = [np.ascontiguousarray(a, dtype=np.float64).reshape(s) for a, s in
           ((x, (B, N + 1, NX)), (u, (B, N, NU)), (yref, (B, N, NY)), (yref_e, (B, NX)))]
    dx = np.empty((B, K, N + 1, NX)) if states else None
    du = np.empty((B, K, N, NU))
    _emu_lib(flavour).emu_jvp_f64(C.byref(cfg), _p(W), _p(act), int(K), *(_p(t) for t in tan), *(_p(a) for a in sol),
                                  _p(dx), _p(du))
    return dx, du
