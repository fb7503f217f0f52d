"""TEST-ONLY: the two references of tests/test_adjoint.py, built on first use next to their sources.

rti_adjoint  -> tests/sens/rti_adjoint.c: the oracle's linearisation and LQR routines with an explicit costate recursion
emu_adjoint  -> tests/sens/emu_adjoint.cpp: the product's qmpc_adjoint_kernel under the lane emulation of tests/emu"""
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
        src = os.path.join(_HERE, "rti_adjoint.c")
        so = _build("librti_adjoint.so",
                    lambda so: ["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-o", so, src, "-lm"],
                    [src, os.path.join(_ROOT, "oracle", "qmpc_oracle.c")])
        _LIBS["oracle"] = C.CDLL(so)
    return _LIBS["oracle"]


def _emu_lib(flavour):
    key = "emu_" + flavour
    if key not in _LIBS:
        defs, _ = emu.FLAVOURS[flavour]
        src = os.path.join(_HERE, "emu_adjoint.cpp")
        emu_dir = os.path.join(_ROOT, "tests", "emu")
        csrc = os.path.join(_ROOT, "mpc_quad_ros_b200", "csrc")
        srcs = [src, os.path.join(emu_dir, "emu_cuda.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                             if f.endswith((".cuh", ".h"))]
        so = _build("libemu_adjoint%s.so" % ("_" + flavour if flavour else ""),
                    lambda so: ["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", emu_dir] + defs +
                               ["-o", so, src], srcs)
        _LIBS[key] = C.CDLL(so)
    return _LIBS[key]


def rti_adjoint(quad, dt, N, xit, uit, act, x_bar=None, u_bar=None, gp=None, alpha=None, Wd=orc.W_DIAG, Wed=orc.WE_DIAG):
    """Reverse mode of oracle.rti_step's result w.r.t. x0 and the reference at the explicit active set act [4N], for the
    cotangents x_bar [N+1,13], u_bar [N,4] (None = zero).  xit, uit: the PRE-solve iterate.
    returns (x0_bar [13], yref_bar [N,17], yref_e_bar [13])"""
    assert xit.shape == (N + 1, NX) and uit.shape == (N, NU)
    act = np.ascontiguousarray(act, dtype=np.uint8).reshape(N * NU)
    x0b, yb, yeb = np.empty(NX), np.empty((N, NX + NU)), np.empty(NX)
    c = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    M = gp.M if gp is not None else 0
    args = [c(a) for a in (quad, alpha, Wd, Wed, xit, uit, x_bar, u_bar)]       # alive until the call returns
    quad, alpha, Wd, Wed, xit, uit, x_bar, u_bar = args
    ok = _oracle_lib().orc_rti_adjoint(_p(quad), C.c_double(dt), N, M, _p(gp.X if gp else None),
                                       _p(gp.theta if gp else None), _p(alpha), _p(Wd), _p(Wed), _p(xit), _p(uit),
                                       _p(act), _p(x_bar), _p(u_bar), _p(x0b), _p(yb), _p(yeb))
    assert ok == 1, "non-positive-definite factorisation in orc_rti_adjoint"
    return x0b, yb, yeb


def emu_adjoint(cfg, r, x_bar=None, u_bar=None, outputs=(True, True, True), flavour=""):
    """qmpc_eval_adjoint emulated on the tiles and active set of an fp64 emu.solve result `r`; x_bar [B,N+1,13],
    u_bar [B,N,4] or None; outputs: which of (x0_bar, yref_bar, yref_e_bar) to ask for (the others come back None).
    returns (x0_bar [B,13], yref_bar [B,N,17], yref_e_bar [B,13])"""
    B, N = cfg.batch, cfg.n_nodes
    W, act = np.ascontiguousarray(r["W"]), np.ascontiguousarray(r["act"], dtype=np.uint8)
    assert W.dtype == np.float64 and W.shape[-1] == emu.FLAVOURS[flavour][1]
    out = [np.empty(s) if want else None for s, want in zip(((B, NX), (B, N, NX + NU), (B, NX)), outputs)]
    xb = None if x_bar is None else np.ascontiguousarray(x_bar, dtype=np.float64).reshape(B, N + 1, NX)
    ub = None if u_bar is None else np.ascontiguousarray(u_bar, dtype=np.float64).reshape(B, N, NU)
    _emu_lib(flavour).emu_adjoint_f64(C.byref(cfg), _p(W), _p(act), _p(xb), _p(ub), *(_p(o) for o in out))
    return tuple(out)
