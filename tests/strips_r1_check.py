"""Shared by the strip R1 tests: the merged DynamicTileEncode streams of a strip set against the oracle, or against one
context coding the whole image."""
from oracle_py import Oracle
from parity import _eq
from yaik_b200 import capi


def r1_stage(mode3):
    return capi.STAGE_RANGEDYN3 if mode3 else capi.STAGE_RANGEDYN


def oracle_r1(planes, mode3):
    """Oracle.range_dyn of R, G, B on the whole image after the alpha stage (RGBA) and the gradient cascade."""
    o = Oracle(planes)
    if planes.shape[0] == 4:
        assert o.alpha() is not None
    o.gradient_cascade()
    out = [o.range_dyn(n, mode3=mode3) for n in range(3)]
    o.close()
    return out


def whole_image_r1(ctx, planes, mode3):
    """The same streams from one context: yk_analyze(ALPHA | GRADIENT | RANGE1D | RANGEDYN) on the whole image."""
    ctx.set_image(planes, 0)
    ctx.analyze((capi.STAGE_ALPHA if planes.shape[0] == 4 else 0) | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D | r1_stage(mode3))
    return [ctx.range_dyn(n, mode3=mode3) for n in range(3)]


def check_r1(merged, wants, what="strips"):
    for n in range(3):
        got, want = merged["r1"][n], wants[n]
        assert got["constraint"] == want["constraint"], (what, n, got["constraint"], want["constraint"])
        _eq(got["defs"], want["defs"], f"{what}: R1 defs plane {n}")
        assert got["n_nibbles"] == want["n_nibbles"], (what, n, got["n_nibbles"], want["n_nibbles"])
        _eq(got["nibbles"], want["nibbles"], f"{what}: R1 nibbles plane {n}")
