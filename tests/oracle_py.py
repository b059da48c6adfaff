"""TEST INFRASTRUCTURE: ctypes binding of oracle/_build/libyaik_oracle.so (the plain-C restatement of the
reference's hot path, oracle/yaik_oracle.c).  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this; the product path never does."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "oracle", "_build", "libyaik_oracle.so")

PASS_ORDER = [(4, 4), (4, 3), (3, 4), (3, 3), (3, 2), (2, 3), (2, 2)]     # EC.cpp:9057-9093
_SWZ = {(4, 4): (64, 64), (4, 3): (64, 64), (3, 4): (64, 64), (3, 3): (64, 64), (3, 2): (64, 32), (2, 3): (32, 64), (2, 2): (32, 32)}


def bitmap_bytes(w, h, shx, shy):
    bw, bh = _SWZ[(shx, shy)]
    bits = (bw >> shx) * (bh >> shy)
    return ((w + bw - 1) // bw) * ((h + bh - 1) // bh) * bits // 8


def build():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(os.path.join(ROOT, "oracle", "yaik_oracle.c")):
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "oracle"], check=True)


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB)
        L.yko_create.restype = C.c_void_p
        L.yko_create.argtypes = [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.yko_destroy.argtypes = [C.c_void_p]
        L.yko_state_plane.restype = C.POINTER(C.c_int32)
        L.yko_state_plane.argtypes = [C.c_void_p, C.c_int]
        for f in ("yko_alpha_reject", "yko_gradient_pass", "yko_range1d", "yko_range_dyn", "yko_dyn_table", "yko_sample_down", "yko_range_dyn_plane"):
            getattr(L, f).restype = C.c_int
        _lib = L
    return _lib


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class Oracle:
    def __init__(self, planes: np.ndarray):
        planes = np.ascontiguousarray(planes, dtype=np.int32)
        self.c, self.h, self.w = planes.shape
        self._planes = planes
        ptrs = (C.c_void_p * self.c)(*[planes[i].ctypes.data for i in range(self.c)])
        self.ctx = lib().yko_create(self.w, self.h, self.c, ptrs)
        assert self.ctx

    def close(self):
        if self.ctx:
            lib().yko_destroy(C.c_void_p(self.ctx))
            self.ctx = None

    __del__ = close

    def alpha(self):
        bm = np.zeros(max(1, (self.w // 16) * (self.h // 16) // 8 + 1), np.uint8)
        nb, rem, wrote = C.c_int(), C.c_int(), C.c_int()
        bound = (C.c_int * 4)(); cb = (C.c_int * 4)()
        rc = lib().yko_alpha_reject(C.c_void_p(self.ctx), _p(bm), C.byref(nb), bound, C.byref(rem), C.byref(wrote), cb)
        if rc != 0:
            return None
        return dict(bitmap=bm[:nb.value].copy(), bound=list(bound), remaining=rem.value, wrote=wrote.value,
                    chunk_bbox=list(cb) if wrote.value else [])

    def gradient_pass(self, shx, shy, reject=3):
        bm = np.zeros(bitmap_bytes(self.w, self.h, shx, shy) + 8, np.uint8)
        rgb = np.zeros(3 * (self.w // (1 << shx) + 1) * (self.h // (1 << shy) + 1) + 8, np.uint8)
        nb, nr, done = C.c_int(), C.c_int(), C.c_int()
        bbox = (C.c_int * 4)()
        rc = lib().yko_gradient_pass(C.c_void_p(self.ctx), reject, shx, shy, _p(bm), C.byref(nb), _p(rgb), C.byref(nr), bbox, C.byref(done))
        assert rc == 0
        return dict(bitmap=bm[:nb.value].copy(), rgb=rgb[:nr.value].copy(), bbox=list(bbox), tiledone=done.value)

    def gradient_cascade(self, reject=3):
        return [self.gradient_pass(sx, sy, reject=reject) for sx, sy in PASS_ORDER]

    def range1d(self, plane, want_debug=False):
        idx = np.zeros(self.w * self.h + 8, np.uint8)
        typ = np.zeros(3 * (self.w // 8 + 1) * (self.h // 8 + 1) + 8, np.uint8)
        dbg = np.zeros((self.h, self.w), np.int32) if want_debug else None
        ni, nt = C.c_int(), C.c_int()
        rc = lib().yko_range1d(C.c_void_p(self.ctx), plane, _p(idx), C.byref(ni), _p(typ), C.byref(nt), _p(dbg) if want_debug else None)
        assert rc == 0
        return dict(idx=idx[:ni.value].copy(), type=typ[:nt.value].copy(), debug=dbg)

    def range_dyn(self, plane, mode3=False, want_dst=False, dst_fill=-1):
        nt = (self.w // 8) * (self.h // 8)
        nib = np.zeros(nt * 32 + 8, np.uint8)
        defs = np.zeros(nt + 8, np.uint16)
        dst = np.full((self.h, self.w), dst_fill, np.int32) if want_dst else None
        nn, nd = C.c_int(), C.c_int()
        cons = (C.c_int * 4)()
        rc = lib().yko_range_dyn(C.c_void_p(self.ctx), plane, int(mode3), _p(nib), C.byref(nn), _p(defs), C.byref(nd),
                                 _p(dst) if want_dst else None, cons)
        assert rc == 0
        return dict(nibbles=nib[:(nn.value + 1) // 2].copy(), n_nibbles=nn.value, defs=defs[:nd.value].copy(), dst=dst,
                    constraint=list(cons))

    def chroma(self, cfg=(1, 0, 1, 0), modes=(2, 2), dst_fill=-1000):
        """The chroma pipeline of Convert() (EC.cpp:9539-9545): RGB -> YCoCg, SampleDown of Co / Cg as configured
        (cfg = halfCoW, halfCoH, halfCgW, halfCgH; modes = EDownSample of Co, Cg), DynamicTileEncode of Y (4 bit allowed),
        Co (4 bit allowed) and Cg (3 bit only).  Returns the planes and the three coded streams."""
        h, w = self.h, self.w
        Y = np.zeros((h, w), np.int32); Co = np.zeros((h, w), np.int32); Cg = np.zeros((h, w), np.int32)
        lib().yko_rgb_to_ycocg(C.c_void_p(self.ctx), _p(Y), _p(Co), _p(Cg))
        work = []
        for src, hx, hy, mode in ((Co, cfg[0], cfg[1], modes[0]), (Cg, cfg[2], cfg[3], modes[1])):
            if hx or hy:
                d = np.zeros((h // 2 if hy else h, w // 2 if hx else w), np.int32)
                assert lib().yko_sample_down(_p(src), w, h, int(hx), int(hy), int(mode), _p(d)) == 0
            else:
                d = src.copy()
            work.append(d)
        out = dict(Y=Y, Co=Co, Cg=Cg, workCo=work[0], workCg=work[1], coded=[])
        for src, m3, chroma, hx, hy in ((Y, 0, 0, 0, 0), (work[0], 0, 1, cfg[0], cfg[1]), (work[1], 1, 1, cfg[2], cfg[3])):
            ph, pw = src.shape
            nt = (pw // 8) * (ph // 8)
            nib = np.zeros(nt * 32 + 8, np.uint8); defs = np.zeros(nt + 8, np.uint16)
            dst = np.full((h, w), dst_fill, np.int32)
            nn, nd = C.c_int(), C.c_int(); cons = (C.c_int * 4)()
            rc = lib().yko_range_dyn_plane(C.c_void_p(self.ctx), _p(src), pw, ph, m3, chroma, int(hx), int(hy), _p(nib), C.byref(nn),
                                           _p(defs), C.byref(nd), _p(dst), cons)
            assert rc == 0
            out["coded"].append(dict(nibbles=nib[:(nn.value + 1) // 2].copy(), n_nibbles=nn.value, defs=defs[:nd.value].copy(), dst=dst,
                                     constraint=list(cons)))
        return out

    def state(self, which):
        n = (self.w + 1) * (self.h + 1) if 5 <= which <= 7 else self.w * self.h
        p = lib().yko_state_plane(C.c_void_p(self.ctx), which)
        return np.ctypeslib.as_array(p, shape=(n,)).copy()


def dyn_table(mn, mx, mode):
    lut = (C.c_int * 16)()
    b, r = C.c_int(), C.c_int()
    n = lib().yko_dyn_table(mn, mx, mode, lut, C.byref(b), C.byref(r))
    return list(lut)[:n], b.value, r.value
