"""Run by tests/test_emulated_strips_r1.py in a subprocess with libasan preloaded: strip sets with DynamicTileEncode through
the AddressSanitizer build of the emulated library, every context exactly as large as its strip.  A read of a strip's
sample, mask or cell row at the image's y instead of the strip's runs past the allocation and aborts the process."""
import sys

import numpy as np

import cases
from strips_r1_check import check_r1, oracle_r1
from yaik_b200 import capi, strips
from yaik_b200.synth import make_image, SEED_BASE

lib = capi.load_library(sys.argv[1])
alpha = np.full((128, 128), 255, np.int32)
alpha[:16] = 0
alpha[:, :8] = 0
for planes, n, mode3 in ((cases._patchy(64, 200, 46, 4, 3), 3, False),
                         (cases._with_alpha(make_image(128, 128, 3, SEED_BASE + 20), alpha), 2, True)):
    c, h, w = planes.shape
    rows = strips.strip_rows(h, n)
    ctxs = [capi.Context(w, sh, planes=c, slots=1, lib=lib) for _, sh in rows]
    merged = strips.LocalTransport(ctxs).run(planes, n_strips=n, r1=capi.STAGE_RANGEDYN3 if mode3 else capi.STAGE_RANGEDYN)
    check_r1(merged, oracle_r1(planes, mode3))
    for ctx in ctxs:
        ctx.close()
print("asan strips r1 cases ok")
