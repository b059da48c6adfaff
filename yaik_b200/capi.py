"""ctypes binding of the C ABI declared in include/yaik_b200.h (libyaik_b200.so, built by yaik_b200/build.py with
nvcc for sm_100a).  This is the same stub a maintainer of the reference would write for its FFI
(INTEGRATION.md shows the C++ one); Python is only the test/bench driver here.

There is no CPU fallback: if the CUDA library is missing or no device is present, loading/creating fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libyaik_b200.so")

PASS_ORDER = [(4, 4), (4, 3), (3, 4), (3, 3), (3, 2), (2, 3), (2, 2)]      # EC.cpp:9057-9093
SWIZZLE = {(4, 4): (64, 64), (4, 3): (64, 64), (3, 4): (64, 64), (3, 3): (64, 64), (3, 2): (64, 32), (2, 3): (32, 64), (2, 2): (32, 32)}

STAGE_ALPHA, STAGE_GRADIENT, STAGE_RANGE1D, STAGE_RANGEDYN, STAGE_RANGEDYN3 = 1, 2, 4, 8, 16

EXPORTS = [
    "yk_abi_version", "yk_error_string", "yk_last_cuda_error", "yk_device_count", "yk_create", "yk_destroy",
    "yk_set_stream", "yk_sync", "yk_set_analysis_ctas", "yk_sm_count", "yk_host_alloc", "yk_host_free", "yk_set_image", "yk_set_image_device", "yk_set_upload_format",
    "yk_set_image_interleaved", "yk_set_image_interleaved_device",
    "yk_device_plane", "yk_reset_state", "yk_reset_states", "yk_analyze", "yk_alpha_reject", "yk_prepare_quad_smooth",
    "yk_gradient_pass", "yk_range1d", "yk_range_dyn", "yk_chroma_prepare", "yk_chroma_plane", "yk_range_dyn_chroma", "yk_download_state", "yk_fetch_all", "yk_result_bytes", "yk_launch_count",
    "yk_profile", "yk_profile_read",
    "yk_strip_config", "yk_strip_halo_ptrs", "yk_strip_phase", "yk_strip_set_peers", "yk_strip_run", "yk_strips_link", "yk_strips_run", "yk_alpha_kept", "yk_alpha_assemble",
    "yk_strip_range_dyn", "yk_strip_run_stages", "yk_strips_run_stages",
    "yk_ipc_export", "yk_ipc_open", "yk_ipc_close", "yk_copy_async", "yk_copy_to_host", "yk_copy_from_host",
    "yk_palette_create", "yk_palette_destroy", "yk_palette_reset", "yk_palette_compress",
    "yk_chunk_file_header", "yk_chunk_mipm", "yk_chunk_gtil", "yk_chunk_1dtl", "yk_chunk_plnt", "yk_chunk_end",
]

COMPRESS_FN = C.CFUNCTYPE(C.c_size_t, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int)


class Results(C.Structure):
    """yk_results of include/yaik_b200.h (pointers into the context's pinned arena)."""
    _fields_ = [("bitmap", C.c_void_p * 7), ("bitmapBytes", C.c_int * 7), ("rgb", C.c_void_p * 7), ("rgbBytes", C.c_int * 7),
                ("tileDone", C.c_int * 7), ("bbox", (C.c_int * 4) * 7),
                ("r2Idx", C.c_void_p * 3), ("r2Type", C.c_void_p * 3), ("r2IdxBytes", C.c_int), ("r2TypeBytes", C.c_int),
                ("alphaValid", C.c_int), ("alphaBitmap", C.c_void_p), ("alphaBitmapBytes", C.c_int), ("alphaBound", C.c_int * 4),
                ("alphaRemaining", C.c_int), ("alphaWroteChunk", C.c_int), ("alphaChunkBBox", C.c_int * 4)]


class StripHalo(C.Structure):
    """yk_strip_halo of include/yaik_b200.h."""
    _fields_ = [("haloIn", C.c_void_p), ("haloBytes", C.c_size_t),
                ("pixelRowInOffset", C.c_size_t), ("pixelRowBytes", C.c_size_t), ("pixelRowStride", C.c_size_t),
                ("touchInTopOffset", C.c_size_t), ("touchInBottomOffset", C.c_size_t), ("touchBytes", C.c_size_t),
                ("pixelRowOut", C.c_void_p * 3), ("planeRowBytes", C.c_size_t),
                ("touchOutTop", C.c_void_p), ("touchOutBottom", C.c_void_p)]


class YaikError(RuntimeError):
    def __init__(self, code, what, detail=""):
        super().__init__(f"{what}: error {code} {detail}")
        self.code = code


def bitmap_bytes(w, h, shx, shy):
    bw, bh = SWIZZLE[(shx, shy)]
    return ((w + bw - 1) // bw) * ((h + bh - 1) // bh) * ((bw >> shx) * (bh >> shy)) // 8


def load_library(path: str | None = None):
    path = path or os.environ.get("YK_LIB") or LIB_PATH      # YK_LIB: developer override for A/B builds of the same sources
    if not os.path.exists(path):
        raise ImportError(f"{path} is missing: build it with `python -m yaik_b200.build` (nvcc, sm_100a). "
                          "yaik_b200 has no CPU fallback.")
    L = C.CDLL(path)
    L.yk_error_string.restype = C.c_char_p
    L.yk_last_cuda_error.restype = C.c_char_p
    L.yk_host_alloc.restype = C.c_void_p
    L.yk_host_alloc.argtypes = [C.c_size_t]
    L.yk_host_free.argtypes = [C.c_void_p]
    L.yk_device_plane.restype = C.c_void_p
    L.yk_device_plane.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.yk_launch_count.restype = C.c_longlong
    L.yk_launch_count.argtypes = [C.c_void_p]
    L.yk_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
    L.yk_destroy.argtypes = [C.c_void_p]
    L.yk_destroy.restype = None
    L.yk_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    L.yk_sync.argtypes = [C.c_void_p]
    L.yk_set_analysis_ctas.argtypes = [C.c_void_p, C.c_int]
    L.yk_sm_count.argtypes = [C.c_void_p]
    L.yk_set_image.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int]
    L.yk_set_image_device.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int]
    L.yk_set_image_interleaved.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int]
    L.yk_set_image_interleaved_device.argtypes = L.yk_set_image_interleaved.argtypes
    L.yk_reset_state.argtypes = [C.c_void_p, C.c_int]
    L.yk_set_upload_format.argtypes = [C.c_void_p, C.c_int]
    L.yk_reset_states.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.yk_analyze.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
    L.yk_prepare_quad_smooth.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.yk_alpha_reject.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                  C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_gradient_pass.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                   C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_range1d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    L.yk_range_dyn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int),
                               C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]
    L.yk_chroma_prepare.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_chroma_plane.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_range_dyn_chroma.argtypes = L.yk_range_dyn.argtypes
    L.yk_download_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_void_p, C.POINTER(C.c_void_p)]
    L.yk_result_bytes.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_longlong)]
    L.yk_fetch_all.argtypes = [C.c_void_p, C.c_int, C.POINTER(Results)]
    L.yk_strip_config.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.yk_strip_halo_ptrs.argtypes = [C.c_void_p, C.c_int, C.POINTER(StripHalo)]
    L.yk_strip_phase.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.yk_strip_set_peers.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.yk_strip_run.argtypes = [C.c_void_p, C.c_int, C.c_int]
    L.yk_strips_link.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int]
    L.yk_strips_run.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int]
    L.yk_strip_range_dyn.argtypes = [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
    L.yk_strip_run_stages.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.yk_strips_run_stages.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_int]
    L.yk_alpha_kept.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_alpha_assemble.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_int, C.POINTER(C.c_int),
                                    C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.yk_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
    L.yk_ipc_open.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]
    L.yk_ipc_close.argtypes = [C.c_void_p, C.c_void_p]
    L.yk_copy_async.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.yk_copy_to_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.yk_copy_from_host.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
    L.yk_palette_create.restype = C.c_void_p
    L.yk_palette_create.argtypes = [C.c_int]
    L.yk_palette_destroy.restype = None
    L.yk_palette_destroy.argtypes = [C.c_void_p]
    L.yk_palette_reset.restype = None
    L.yk_palette_reset.argtypes = [C.c_void_p]
    L.yk_palette_compress.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(C.c_int)]
    szp = C.POINTER(C.c_size_t)
    L.yk_chunk_file_header.argtypes = [C.c_void_p, C.c_size_t, szp, C.c_int, C.c_int, C.c_int]
    L.yk_chunk_mipm.argtypes = [C.c_void_p, C.c_size_t, szp, C.POINTER(C.c_int), C.c_void_p, C.c_int]
    L.yk_chunk_gtil.argtypes = [C.c_void_p, C.c_size_t, szp, C.c_void_p, COMPRESS_FN, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int),
                                C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
    L.yk_chunk_1dtl.argtypes = [C.c_void_p, C.c_size_t, szp, COMPRESS_FN, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int]
    L.yk_chunk_plnt.argtypes = [C.c_void_p, C.c_size_t, szp, COMPRESS_FN, C.c_void_p, C.POINTER(C.c_int), C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                C.c_int, C.c_int, C.c_int]
    L.yk_chunk_end.argtypes = [C.c_void_p, C.c_size_t, szp]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Context:
    """One yk_ctx: a GPU, `slots` image slots of up to max_w x max_h."""

    def __init__(self, max_w, max_h, planes=4, slots=1, device=0, lib=None, lib_path=None):
        self.L = lib or load_library(lib_path)
        self.ctx = C.c_void_p()
        rc = self.L.yk_create(C.byref(self.ctx), device, max_w, max_h, planes, slots)
        if rc:
            self.ctx = None
            raise YaikError(rc, "yk_create", self.L.yk_last_cuda_error().decode())
        self._keep = {}
        self.dims = {}

    def close(self):
        if getattr(self, "ctx", None):
            self.L.yk_destroy(self.ctx)
            self.ctx = None

    __del__ = close

    def _ck(self, rc, what):
        if rc:
            raise YaikError(rc, what, self.L.yk_error_string(rc).decode() + " " + self.L.yk_last_cuda_error().decode())

    def set_stream(self, cuda_stream: int):
        self._ck(self.L.yk_set_stream(self.ctx, C.c_void_p(cuda_stream)), "yk_set_stream")

    def set_analysis_ctas(self, ctas: int):
        self._ck(self.L.yk_set_analysis_ctas(self.ctx, ctas), "yk_set_analysis_ctas")

    def sm_count(self) -> int:
        return int(self.L.yk_sm_count(self.ctx))

    def sync(self):
        self._ck(self.L.yk_sync(self.ctx), "yk_sync")

    def set_image(self, planes: np.ndarray, slot=0):
        planes = np.ascontiguousarray(planes, dtype=np.int32)
        c, h, w = planes.shape
        ptrs = (C.c_void_p * c)(*[planes[i].ctypes.data for i in range(c)])
        self._keep[slot] = planes
        self.dims[slot] = (c, h, w)
        self._ck(self.L.yk_set_image(self.ctx, slot, ptrs, c, w, h), "yk_set_image")
        self.sync()      # the source array may be pageable numpy memory

    def set_upload_format(self, packed_u8: bool):
        self._ck(self.L.yk_set_upload_format(self.ctx, int(packed_u8)), "yk_set_upload_format")

    def set_image_ptrs(self, host_ptrs, c, w, h, slot=0):
        """Pinned host plane pointers (yk_host_alloc); asynchronous."""
        ptrs = (C.c_void_p * c)(*host_ptrs)
        self.dims[slot] = (c, h, w)
        self._ck(self.L.yk_set_image(self.ctx, slot, ptrs, c, w, h), "yk_set_image")

    def set_image_device(self, dev_ptrs, c, w, h, slot=0):
        ptrs = (C.c_void_p * c)(*dev_ptrs)
        self.dims[slot] = (c, h, w)
        self._ck(self.L.yk_set_image_device(self.ctx, slot, ptrs, c, w, h), "yk_set_image_device")

    def set_image_interleaved(self, pixels: np.ndarray, n_planes=None, slot=0):
        """An H x W x C uint8 image (C = 3 RGB or 4 RGBA; the row stride may exceed W * C) from host memory."""
        if pixels.dtype != np.uint8 or pixels.ndim != 3 or pixels.strides[1:] != (pixels.shape[2], 1):
            pixels = np.ascontiguousarray(pixels, dtype=np.uint8)
        h, w, ch = pixels.shape
        self._keep[slot] = pixels
        self.set_image_interleaved_ptr(pixels.ctypes.data, pixels.strides[0], ch, n_planes or ch, w, h, slot)
        self.sync()      # the source array may be pageable numpy memory

    def set_image_interleaved_ptr(self, ptr, row_bytes, channels, n_planes, w, h, slot=0):
        """Interleaved rows at a host address (pinned from yk_host_alloc: asynchronous until the next synchronising call)."""
        self.dims[slot] = (n_planes, h, w)
        self._ck(self.L.yk_set_image_interleaved(self.ctx, slot, C.c_void_p(ptr), row_bytes, channels, n_planes, w, h), "yk_set_image_interleaved")

    def set_image_interleaved_device(self, dev_ptr, row_bytes, channels, n_planes, w, h, slot=0):
        """Interleaved rows in device memory, read by a kernel on the context's stream (the buffer is not kept)."""
        self.dims[slot] = (n_planes, h, w)
        self._ck(self.L.yk_set_image_interleaved_device(self.ctx, slot, C.c_void_p(dev_ptr), row_bytes, channels, n_planes, w, h),
                 "yk_set_image_interleaved_device")

    def device_plane(self, slot, p):
        return self.L.yk_device_plane(self.ctx, slot, p)

    def reset_state(self, slot=0):
        self._ck(self.L.yk_reset_state(self.ctx, slot), "yk_reset_state")

    def reset_states(self, slot0, n_slots):
        self._ck(self.L.yk_reset_states(self.ctx, slot0, n_slots), "yk_reset_states")

    def analyze(self, stages, slot0=0, n_slots=1, reject=3):
        self._ck(self.L.yk_analyze(self.ctx, slot0, n_slots, stages, reject), "yk_analyze")

    def prepare_quad_smooth(self, slot=0, reject=3):
        self._ck(self.L.yk_prepare_quad_smooth(self.ctx, slot, reject), "yk_prepare_quad_smooth")

    def alpha_reject(self, slot=0):
        c, h, w = self.dims[slot]
        cap = ((w + 15) // 16) * ((h + 15) // 16) // 8 + 8
        bm = np.zeros(cap, np.uint8)
        nb, rem, wrote = C.c_int(), C.c_int(), C.c_int()
        bound = (C.c_int * 4)(); cb = (C.c_int * 4)()
        self._ck(self.L.yk_alpha_reject(self.ctx, slot, _p(bm), cap, C.byref(nb), bound, C.byref(rem), C.byref(wrote), cb), "yk_alpha_reject")
        return dict(bitmap=bm[:nb.value].copy(), bound=list(bound), remaining=rem.value, wrote=wrote.value,
                    chunk_bbox=list(cb) if wrote.value else [])

    def gradient_pass(self, shx, shy, slot=0, reject=3):
        c, h, w = self.dims[slot]
        capb = bitmap_bytes(w, h, shx, shy) + 8
        capr = 3 * (w // (1 << shx) + 1) * (h // (1 << shy) + 1) + 8
        bm = np.zeros(capb, np.uint8); rgb = np.zeros(capr, np.uint8)
        nb, nr, done = C.c_int(), C.c_int(), C.c_int()
        bbox = (C.c_int * 4)()
        self._ck(self.L.yk_gradient_pass(self.ctx, slot, reject, shx, shy, _p(bm), capb, C.byref(nb), _p(rgb), capr, C.byref(nr), bbox, C.byref(done)), "yk_gradient_pass")
        return dict(bitmap=bm[:nb.value].copy(), rgb=rgb[:nr.value].copy(), bbox=list(bbox), tiledone=done.value)

    def range1d(self, plane, slot=0):
        c, h, w = self.dims[slot]
        capi, capt = w * h + 8, 3 * (w // 8 + 1) * (h // 8 + 1) + 8
        idx = np.zeros(capi, np.uint8); typ = np.zeros(capt, np.uint8)
        ni, nt = C.c_int(), C.c_int()
        self._ck(self.L.yk_range1d(self.ctx, slot, plane, _p(idx), capi, C.byref(ni), _p(typ), capt, C.byref(nt)), "yk_range1d")
        return dict(idx=idx[:ni.value].copy(), type=typ[:nt.value].copy())

    def range_dyn(self, plane, mode3=False, slot=0, want_dst=False, dst_fill=-1):
        c, h, w = self.dims[slot]
        nt = (w // 8) * (h // 8)
        capn = nt * 32 + 8
        nib = np.zeros(capn, np.uint8); defs = np.zeros(nt + 8, np.uint16)
        dst = np.full((h, w), dst_fill, np.int32) if want_dst else None
        nn, nd = C.c_int(), C.c_int()
        cons = (C.c_int * 4)()
        self._ck(self.L.yk_range_dyn(self.ctx, slot, plane, int(mode3), _p(nib), capn, C.byref(nn), _p(defs), nt + 8, C.byref(nd), cons, _p(dst)), "yk_range_dyn")
        return dict(nibbles=nib[:(nn.value + 1) // 2].copy(), n_nibbles=nn.value, defs=defs[:nd.value].copy(), dst=dst, constraint=list(cons))

    def chroma(self, cfg=(1, 0, 1, 0), modes=(2, 2), slot=0, dst_fill=-1000, planes=True):
        """The chroma pipeline of Convert() (EC.cpp:9539-9545): yk_chroma_prepare, then DynamicTileEncode of Y, workCo and
        workCg with the reference's mode3BitOnly = 0, 0, 1.  cfg = halfCoW, halfCoH, halfCgW, halfCgH; modes = EDownSample."""
        c, h, w = self.dims[slot]
        half = (C.c_int * 4)(*[int(v) for v in cfg]); dm = (C.c_int * 2)(*[int(v) for v in modes])
        self._ck(self.L.yk_chroma_prepare(self.ctx, slot, half, dm), "yk_chroma_prepare")
        out = dict(coded=[])
        for which, key in enumerate(("Y", "workCo", "workCg")):
            pw, ph = C.c_int(), C.c_int()
            self._ck(self.L.yk_chroma_plane(self.ctx, slot, which, None, C.byref(pw), C.byref(ph)), "yk_chroma_plane")
            if planes:
                a = np.zeros((ph.value, pw.value), np.int32)
                self._ck(self.L.yk_chroma_plane(self.ctx, slot, which, _p(a), None, None), "yk_chroma_plane")
                out[key] = a
            nt = (pw.value // 8) * (ph.value // 8)
            capn = nt * 32 + 8
            nib = np.zeros(capn, np.uint8); defs = np.zeros(nt + 8, np.uint16)
            dst = np.full((h, w), dst_fill, np.int32)
            nn, nd = C.c_int(), C.c_int()
            cons = (C.c_int * 4)()
            self._ck(self.L.yk_range_dyn_chroma(self.ctx, slot, which, int(which == 2), _p(nib), capn, C.byref(nn), _p(defs), nt + 8, C.byref(nd),
                                                cons, _p(dst)), "yk_range_dyn_chroma")
            out["coded"].append(dict(nibbles=nib[:(nn.value + 1) // 2].copy(), n_nibbles=nn.value, defs=defs[:nd.value].copy(), dst=dst,
                                     constraint=list(cons)))
        return out

    def download_state(self, slot=0, recon=True):
        c, h, w = self.dims[slot]
        smooth = np.zeros((h, w), np.int32); mask = np.zeros((h, w), np.int32)
        mst = [np.zeros((h, w), np.int32) for _ in range(3)]
        mrgb = [np.zeros((h + 1, w + 1), np.int32) for _ in range(3)]
        rec = [np.zeros((h, w), np.int32) for _ in range(3)] if recon else None
        arr = lambda lst: (C.c_void_p * 3)(*[a.ctypes.data for a in lst])
        self._ck(self.L.yk_download_state(self.ctx, slot, _p(smooth), arr(mst), arr(mrgb), _p(mask), arr(rec) if recon else None), "yk_download_state")
        return dict(smoothMap=smooth, mapSmoothTile=mst, mappedRGB=mrgb, mipmapMask=mask, recon=rec)

    # ---- strips (one large image over several GPUs / contexts) ----
    def strip_config(self, img_h, y0, slot=0):
        self._ck(self.L.yk_strip_config(self.ctx, slot, img_h, y0), "yk_strip_config")

    def strip_halo(self, slot=0) -> "StripHalo":
        h = StripHalo()
        self._ck(self.L.yk_strip_halo_ptrs(self.ctx, slot, C.byref(h)), "yk_strip_halo_ptrs")
        return h

    def strip_set_peers(self, above, below, slot=0):
        self._ck(self.L.yk_strip_set_peers(self.ctx, slot, C.c_void_p(above or 0), C.c_void_p(below or 0)), "yk_strip_set_peers")

    def strip_run(self, slot=0, reject=3, stages=0):
        """One image without the host in the loop; stages = 0, STAGE_RANGEDYN or STAGE_RANGEDYN3 (R1 of an RGB strip)."""
        self._ck(self.L.yk_strip_run_stages(self.ctx, slot, reject, stages), "yk_strip_run_stages")

    def strip_range_dyn(self, mode3=False, bound=None, slot=0):
        """DynamicTileEncode of the strip's rows after phase 0 (range_dyn then returns the strip's part).  bound: the strip
        set's merged alpha box for RGBA (strips.merge_alpha), None for RGB."""
        box = (C.c_int * 4)(*bound) if bound is not None else None
        self._ck(self.L.yk_strip_range_dyn(self.ctx, slot, int(mode3), box), "yk_strip_range_dyn")

    def alpha_kept(self, slot=0):
        """Per-tile alpha results of one strip (or image): kept bytes [th][tw], box of the kept tiles in image coordinates."""
        c, h, w = self.dims[slot]
        tw, th = (w + 15) // 16, (h + 15) // 16
        kept = np.zeros(tw * th, np.uint8)
        a, b, n = C.c_int(), C.c_int(), C.c_int()
        bound = (C.c_int * 4)()
        self._ck(self.L.yk_alpha_kept(self.ctx, slot, _p(kept), kept.size, C.byref(a), C.byref(b), bound, C.byref(n)), "yk_alpha_kept")
        return dict(kept=kept.reshape(th, tw), bound=list(bound), count=n.value)

    def strip_phase(self, phase, slot=0, reject=3):
        self._ck(self.L.yk_strip_phase(self.ctx, slot, phase, reject), "yk_strip_phase")

    def copy_async(self, dst, src, nbytes):
        self._ck(self.L.yk_copy_async(self.ctx, C.c_void_p(dst), C.c_void_p(src), nbytes), "yk_copy_async")

    def copy_to_host(self, dev_src, nbytes) -> np.ndarray:
        out = np.empty(nbytes, np.uint8)
        self._ck(self.L.yk_copy_to_host(self.ctx, _p(out), C.c_void_p(dev_src), nbytes), "yk_copy_to_host")
        return out

    def copy_from_host(self, dev_dst, data: np.ndarray):
        data = np.ascontiguousarray(data).view(np.uint8).ravel()
        self._ck(self.L.yk_copy_from_host(self.ctx, C.c_void_p(dev_dst), _p(data), data.size), "yk_copy_from_host")

    def ipc_export(self, dev_ptr) -> bytes:
        buf = C.create_string_buffer(64)
        self._ck(self.L.yk_ipc_export(C.c_void_p(dev_ptr), buf), "yk_ipc_export")
        return buf.raw

    def ipc_open(self, handle: bytes) -> int:
        out = C.c_void_p()
        self._ck(self.L.yk_ipc_open(self.ctx, handle, C.byref(out)), "yk_ipc_open")
        return out.value

    def ipc_close(self, dev_ptr):
        self._ck(self.L.yk_ipc_close(self.ctx, C.c_void_p(dev_ptr)), "yk_ipc_close")

    def fetch_all(self, slot=0, copy=True):
        """Everything of the last run with one call (yk_fetch_all).  copy=False returns the raw Results struct whose pointers
        lead into the context's pinned arena."""
        r = Results()
        self._ck(self.L.yk_fetch_all(self.ctx, slot, C.byref(r)), "yk_fetch_all")
        if not copy:
            return r

        def arr(ptr, n):
            return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_uint8)), shape=(n,)).copy() if ptr and n else np.zeros(0, np.uint8)
        out = {"passes": [], "r2": [], "alpha": None}
        for p in range(7):
            out["passes"].append(None if not r.bitmap[p] else dict(bitmap=arr(r.bitmap[p], r.bitmapBytes[p]), rgb=arr(r.rgb[p], r.rgbBytes[p]),
                                                                  tiledone=r.tileDone[p], bbox=list(r.bbox[p])))
        for pl in range(3):
            if r.r2Idx[pl]:
                out["r2"].append(dict(idx=arr(r.r2Idx[pl], r.r2IdxBytes), type=arr(r.r2Type[pl], r.r2TypeBytes)))
        if r.alphaValid:
            out["alpha"] = dict(bitmap=arr(r.alphaBitmap, r.alphaBitmapBytes), bound=list(r.alphaBound), remaining=r.alphaRemaining,
                                wrote=r.alphaWroteChunk, chunk_bbox=list(r.alphaChunkBBox) if r.alphaWroteChunk else [])
        return out

    def result_bytes(self, slot=0):
        out = (C.c_longlong * 6)()
        self._ck(self.L.yk_result_bytes(self.ctx, slot, out), "yk_result_bytes")
        return list(out)

    def launch_count(self):
        return int(self.L.yk_launch_count(self.ctx))
