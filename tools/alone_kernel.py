"""Developer tool: yk_k_analyze / yk_k_emit / yk_k_owner timed alone (yk_profile: event pair around each launch) for the
library named by YK_LIB on the bench texture; no result check."""
import sys, os, ctypes as C
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from yaik_b200 import capi
from yaik_b200.synth import make_image, SEED_BASE
lib = capi.load_library(os.environ.get('YK_LIB'))
ctx = capi.Context(2048, 2048, planes=4, slots=1, lib=lib)
ctx.set_upload_format(False)
ctx.set_image(make_image(2048, 2048, 4, SEED_BASE + 1), 0)
st = capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D
for _ in range(5):
    ctx.reset_state(0); ctx.analyze(st); ctx.sync()
lib.yk_profile(ctx.ctx, 1)
for _ in range(40):
    ctx.reset_state(0); ctx.analyze(st); ctx.sync()
a = (C.c_double * 8)(); b = (C.c_longlong * 8)()
lib.yk_profile_read(ctx.ctx, a, b)
print(os.path.basename(os.environ.get('YK_LIB', 'default')), {n: round(a[i] / max(b[i], 1) * 1e3, 2) for i, n in enumerate(["analyze_us", "emit_us", "owner_us"])})
