"""TEST-ONLY: the two references of tests/test_sensitivities.py, built on first use next to their sources.

rti_sens  -> tests/sens/rti_sens.c: the oracle's linearisation and LQR routines, 13 independent LQR solves
emu_sens  -> tests/sens/emu_sens.cpp: the product's qmpc_sens_kernel under the lane emulation of tests/emu"""
import ctypes as C
import os
import subprocess

import numpy as np

from emu import emu
from oracle import oracle as orc

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(os.path.dirname(_HERE))
_LIBS = {}
NX, NU = 13, 4


def _build(name, cmd_of, srcs):
    so = os.path.join(_HERE, name)
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
        subprocess.check_call(cmd_of(so))
    return so


def _oracle_lib():
    if "oracle" not in _LIBS:
        src = os.path.join(_HERE, "rti_sens.c")
        so = _build("librti_sens.so",
                    lambda so: ["gcc", "-O2", "-fPIC", "-std=c11", "-shared", "-o", so, src, "-lm"],
                    [src, os.path.join(_ROOT, "oracle", "qmpc_oracle.c")])
        _LIBS["oracle"] = C.CDLL(so)
    return _LIBS["oracle"]


def _emu_lib(flavour):
    key = "emu_" + flavour
    if key not in _LIBS:
        defs, _ = emu.FLAVOURS[flavour]
        src = os.path.join(_HERE, "emu_sens.cpp")
        emu_dir = os.path.join(_ROOT, "tests", "emu")
        csrc = os.path.join(_ROOT, "mpc_quad_ros_b200", "csrc")
        srcs = [src, os.path.join(emu_dir, "emu_cuda.h")] + [os.path.join(csrc, f) for f in os.listdir(csrc)
                                                             if f.endswith((".cuh", ".h"))]
        so = _build("libemu_sens%s.so" % ("_" + flavour if flavour else ""),
                    lambda so: ["g++", "-std=c++20", "-O2", "-fPIC", "-shared", "-pthread", "-I", emu_dir] + defs +
                               ["-o", so, src], srcs)
        _LIBS[key] = C.CDLL(so)
    return _LIBS[key]


def _p(a):
    return C.c_void_p(0) if a is None else a.ctypes.data_as(C.c_void_p)


def rti_sens(quad, dt, N, xit, uit, act, n_stages=None, gp=None, alpha=None, Wd=orc.W_DIAG, Wed=orc.WE_DIAG,
             states=True):
    """Derivatives of oracle.rti_step's result w.r.t. x0 at the explicit active set act [4N] (0 free, 1 lower, 2 upper).
    xit [(N+1),13], uit [N,4]: the PRE-solve iterate (the linearisation point).
    returns (sens_x [n+1,13,13] or None, sens_u [n,4,13]); column i = derivative w.r.t. x0[i]"""
    n = N if n_stages is None else int(n_stages)
    assert 1 <= n <= N and xit.shape == (N + 1, NX) and uit.shape == (N, NU)
    act = np.ascontiguousarray(act, dtype=np.uint8).reshape(N * NU)
    sx = np.empty((n + 1, NX, NX)) if states else None
    su = np.empty((n, NU, NX))
    c = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    M = gp.M if gp is not None else 0
    ok = _oracle_lib().orc_rti_sens(_p(c(quad)), C.c_double(dt), N, M, _p(gp.X if gp else None),
                                    _p(gp.theta if gp else None), _p(c(alpha)), _p(c(Wd)), _p(c(Wed)), _p(c(xit)),
                                    _p(c(uit)), _p(act), n, _p(sx), _p(su))
    assert ok == 1, "non-positive-definite factorisation in orc_rti_sens"
    return sx, su


def emu_sens(cfg, r, n_stages, states=True, flavour=""):
    """qmpc_eval_sens_x0 emulated on the tiles and active set of an fp64 emu.solve result `r`.
    returns (sens_x [B, n_stages+1, 13, 13] or None, sens_u [B, n_stages, 4, 13])"""
    B = cfg.batch
    W, act = np.ascontiguousarray(r["W"]), np.ascontiguousarray(r["act"], dtype=np.uint8)
    assert W.dtype == np.float64 and W.shape[-1] == emu.FLAVOURS[flavour][1]
    sx = np.empty((B, n_stages + 1, NX, NX)) if states else None
    su = np.empty((B, n_stages, NU, NX))
    _emu_lib(flavour).emu_sens_f64(C.byref(cfg), _p(W), _p(act), int(n_stages), _p(sx), _p(su))
    return sx, su
