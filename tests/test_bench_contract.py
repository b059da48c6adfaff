"""bench.py's contract: the reference arm prints one JSON line with the keys of the result line, the GPU arm refuses to run
(no CPU fallback) when there is no device, and (-m gpu) it times --steps steps and dumps the outputs of the last one."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT, env=env)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["unit"] == "MP/s" and line["higher_is_better"] is True and line["value"] > 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"]


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_has_no_cpu_fallback():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")        # no device, also where the machine has one
    r = _run("--steps", "1", "--warmup", "1", "--no-cpu", "--e2e-steps", "0", "--roofline-steps", "0", timeout=300, env=env)
    assert r.returncode != 0, "bench.py must fail without a CUDA device, not fall back to a CPU path"
    assert not any(l.startswith("{") and '"value"' in l for l in r.stdout.splitlines())


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    """--steps K times K steps, and --dump-outputs writes the streams of the last one in float32 / float64, no file empty,
    at most 64 MB: they equal what a fresh context returns for that texture.  Two streams and seven steps: step 6 runs on
    context 0, slot 3, texture 6 (step i analyses texture i mod 8)."""
    import numpy as np
    from yaik_b200 import capi
    from yaik_b200.synth import make_image, SEED_BASE
    steps = 7
    r = _run("--steps", str(steps), "--streams", "2", "--warmup", "1", "--no-cpu", "--e2e-steps", "0", "--roofline-steps", "0",
             "--no-r1", "--no-other", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["gpu_launches"] == 3 * steps         # three kernels per step (run.kernels_per_step)
    files = sorted(tmp_path.glob("*.npy"))
    assert sum(p.stat().st_size for p in files) <= 64 << 20
    got = {p.stem: np.load(p) for p in files}
    for name, a in got.items():
        assert a.dtype in (np.float32, np.float64) and a.size > 0, name
    c = capi.Context(2048, 2048, planes=4, slots=1)
    try:
        c.set_upload_format(False)
        c.set_image(make_image(2048, 2048, 4, SEED_BASE + 1 + (steps - 1) % 8))
        c.analyze(capi.STAGE_ALPHA | capi.STAGE_GRADIENT | capi.STAGE_RANGE1D)
        want = c.fetch_all(0)
    finally:
        c.close()
    streams, meta = {}, {}
    for k, p in enumerate(want["passes"]):
        streams[f"pass{k}_bitmap"], streams[f"pass{k}_rgb"] = p["bitmap"], p["rgb"]
        meta[f"pass{k}_tiledone_bbox"] = [p["tiledone"], *p["bbox"]]
    for n, q in enumerate(want["r2"]):
        streams[f"r2_idx{n}"], streams[f"r2_type{n}"] = q["idx"], q["type"]
    a = want["alpha"]
    streams["alpha_bitmap"] = a["bitmap"]
    meta["alpha_bound_remaining_wrote_chunk_bbox"] = [*a["bound"], a["remaining"], a["wrote"], *(a["chunk_bbox"] or [0] * 4)]
    meta["stream_lengths"] = [v.size for v in streams.values()]
    assert len(streams) == 7 * 2 + 3 * 2 + 1
    assert set(got) == set(meta) | {n for n, v in streams.items() if v.size}
    for name, v in meta.items():
        assert got[name].dtype == np.float64 and got[name].tolist() == [float(x) for x in v], name
    for name, v in streams.items():
        if v.size:
            assert got[name].dtype == np.float32 and np.array_equal(got[name], v.astype(np.float32)), name
