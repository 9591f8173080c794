"""The batched regularised LDL^T of small KKT systems (cxb_small_ldlt / cxb_small_ldlt_solve) on the two backends
of small_backend.py: "device" (the real kernels of libconex_b200.so) and "emul" (SmallLdlt / SmallLdltSolve of
small_cone_math.cuh compiled for the host with a serial stand-in for the team, tests/emul/emul_ldlt.cc — test
infrastructure only, never part of the product library).
"""
import ctypes as C
import os
import subprocess

import numpy as np

from small_backend import HEADER, ROOT, Backend, vp

EMUL_LDLT_SRC = os.path.join(ROOT, "tests", "emul", "emul_ldlt.cc")
EMUL_LDLT_SO = os.path.join(ROOT, "tests", "emul", "_build", "libemul_ldlt.so")


def build_emul_ldlt():
    os.makedirs(os.path.dirname(EMUL_LDLT_SO), exist_ok=True)
    newest = max(os.path.getmtime(EMUL_LDLT_SRC), os.path.getmtime(HEADER))
    if not os.path.exists(EMUL_LDLT_SO) or os.path.getmtime(EMUL_LDLT_SO) < newest:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", EMUL_LDLT_SO, EMUL_LDLT_SRC])
    return EMUL_LDLT_SO


class LdltBackend(Backend):
    """kind = "emul" | "device"; memory handling as Backend."""

    def __init__(self, kind):
        if kind == "emul":
            self.kind = kind
            self.lib = C.CDLL(build_emul_ldlt())
            self.prefix = "emul_small_"
        else:
            super().__init__(kind)

    def _call_masked(self, name, args, active):
        """name(args..., active): the mask is the last argument on both backends, the stream the first on the
        device."""
        f = getattr(self.lib, self.prefix + name)
        f.restype = C.c_int
        mask = None if active is None else self.upload(np.asarray(active), np.int32)
        args = args + (self.ptr(mask),)
        if self.kind == "device":
            args = (vp(None),) + args
        rc = f(*args)
        assert rc == 0, (name, rc)

    def ldlt(self, K, active=None, L_init=None):
        """K: (batch, N, N) symmetric matrices (only the lower triangles are read). Returns the factors of
        cxb_small_ldlt: (L batch x N x N lower, perm batch x N, signs batch x N, info batch, device handles,
        K as stored afterwards). L_init: initial contents of the factor storage (batch, N, N)."""
        batch, N, _ = K.shape
        kbuf = self.upload(np.stack([k.T for k in K]))  # column-major
        lbuf = self.upload(np.stack([l.T for l in L_init])) if L_init is not None else self.alloc(batch * N * N)
        perm = self.upload(np.full(batch * N, -7), np.int32)
        signs = self.upload(np.full(batch * N, 5.0))
        info = self.upload(np.full(batch, -3), np.int32)
        self._call_masked("ldlt", (C.c_int(batch), C.c_int(N), self.ptr(kbuf), C.c_long(N), C.c_long(N * N),
                                   self.ptr(lbuf), C.c_long(N), C.c_long(N * N), self.ptr(perm), C.c_long(N),
                                   self.ptr(signs), C.c_long(N), self.ptr(info)), active)
        L = self.download(lbuf).reshape(batch, N, N).transpose(0, 2, 1)
        Kafter = self.download(kbuf).reshape(batch, N, N).transpose(0, 2, 1)
        handles = (lbuf, perm, signs)
        return (L, self.download(perm).reshape(batch, N), self.download(signs).reshape(batch, N),
                self.download(info), handles, Kafter)

    def ldlt_solve(self, handles, batch, N, X, active=None):
        lbuf, perm, signs = handles
        x = self.upload(X)
        self._call_masked("ldlt_solve", (C.c_int(batch), C.c_int(N), self.ptr(lbuf), C.c_long(N), C.c_long(N * N),
                                         self.ptr(perm), C.c_long(N), self.ptr(signs), C.c_long(N), self.ptr(x),
                                         C.c_long(N)), active)
        return self.download(x).reshape(batch, N)
