"""Run by tests/test_emulated_interleaved_input.py in a subprocess with libasan preloaded: interleaved loads through the
AddressSanitizer build of the emulated library, from buffers that end exactly at the last pixel's last byte.  Any read
past a caller's buffer, or any out-of-bounds access of the kernels (as emulated), aborts the process."""
import sys

import cases
from interleaved import loader
from parity import check_image
from yaik_b200 import capi

lib = capi.load_library(sys.argv[1])
for name in ("patchy_72x40", "alpha_island128", "mip8_rgb"):
    planes, stages = cases.SMALL_CASES[name]()
    for how, ch, pad, off in (("host", None, 0, 0), ("device", None, 0, 0), ("host", 4, 0, 3), ("device", 4, 5, 1), ("device", None, 2, 15)):
        p, st = (planes[:3], tuple(s for s in stages if s != "alpha")) if ch == 4 else (planes, stages)
        ctx = capi.Context(128, 128, planes=4, slots=1, lib=lib)
        check_image(ctx, p, st, fused=True, load=loader(how, ch, pad, off))
        ctx.close()
print("asan interleaved cases ok")
