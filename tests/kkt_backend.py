"""The batched KKT factorisations at any order N (cxb_small_potrf / cxb_small_ldlt and their blocked kernels
cxb_small_potrf_blocked / cxb_small_ldlt_blocked) on the two backends of small_backend.py: "device" (the real
kernels of libconex_b200.so) and "emul" (BlockedPotrf / BlockedLdlt of small_cone_math.cuh compiled for the host with
a serial stand-in for the team and the plain-loop trailing update, tests/emul/emul_blocked_kkt.cc — test
infrastructure only, never part of the product library).
"""
import ctypes as C
import os
import subprocess

import numpy as np

from ldlt_backend import LdltBackend
from small_backend import HEADER, ROOT

EMUL_SRC = os.path.join(ROOT, "tests", "emul", "emul_blocked_kkt.cc")
EMUL_SO = os.path.join(ROOT, "tests", "emul", "_build", "libemul_blocked_kkt.so")


def build_emul_blocked():
    os.makedirs(os.path.dirname(EMUL_SO), exist_ok=True)
    newest = max(os.path.getmtime(EMUL_SRC), os.path.getmtime(HEADER))
    if not os.path.exists(EMUL_SO) or os.path.getmtime(EMUL_SO) < newest:
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", EMUL_SO, EMUL_SRC])
    return EMUL_SO


class KktBackend(LdltBackend):
    """kind = "emul" (the blocked kernels only) | "device". blocked=True calls cxb_small_*_blocked, False the entry
    points that choose by N."""

    def __init__(self, kind):
        if kind == "emul":
            self.kind = kind
            self.lib = C.CDLL(build_emul_blocked())
            self.prefix = "emul_small_"
        else:
            super().__init__(kind)

    def potrf(self, H, blocked=True, active=None, H_init=None):
        """H: (batch, N, N) symmetric (lower triangles read). Returns (H as stored afterwards, info, device buffer).
        H_init: what the storage of every program holds before the call (default H)."""
        assert blocked or self.kind == "device"
        batch, N, _ = H.shape
        buf = self.upload(np.stack([h.T for h in (H if H_init is None else H_init)]))
        if H_init is not None:  # the programs to factor get H
            host = self.download(buf).reshape(batch, N, N)
            mask = np.ones(batch, bool) if active is None else np.asarray(active, bool)
            host[mask] = np.stack([h.T for h in H])[mask]
            buf = self.upload(host)
        info = self.upload(np.full(batch, -3), np.int32)
        self._call_masked("potrf_blocked" if blocked else "potrf",
                          (C.c_int(batch), C.c_int(N), self.ptr(buf), C.c_long(N), C.c_long(N * N), self.ptr(info)),
                          active)
        return self.download(buf).reshape(batch, N, N).transpose(0, 2, 1), self.download(info), buf

    def ldlt(self, K, active=None, L_init=None, blocked=True):
        """LdltBackend.ldlt through cxb_small_ldlt_blocked (blocked) or cxb_small_ldlt."""
        assert blocked or self.kind == "device"
        batch, N, _ = K.shape
        kbuf = self.upload(np.stack([k.T for k in K]))  # column-major
        lbuf = self.upload(np.stack([l.T for l in L_init])) if L_init is not None else self.alloc(batch * N * N)
        perm = self.upload(np.full(batch * N, -7), np.int32)
        signs = self.upload(np.full(batch * N, 5.0))
        info = self.upload(np.full(batch, -3), np.int32)
        self._call_masked("ldlt_blocked" if blocked else "ldlt",
                          (C.c_int(batch), C.c_int(N), self.ptr(kbuf), C.c_long(N), C.c_long(N * N), self.ptr(lbuf),
                           C.c_long(N), C.c_long(N * N), self.ptr(perm), C.c_long(N), self.ptr(signs), C.c_long(N),
                           self.ptr(info)), active)
        L = self.download(lbuf).reshape(batch, N, N).transpose(0, 2, 1)
        Kafter = self.download(kbuf).reshape(batch, N, N).transpose(0, 2, 1)
        return (L, self.download(perm).reshape(batch, N), self.download(signs).reshape(batch, N),
                self.download(info), (lbuf, perm, signs), Kafter)
