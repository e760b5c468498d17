"""The driver's bench.py contract: one JSON line with the required keys (checked on CPU with synthetic numbers)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_result_line_has_every_required_key():
    from bench_common import result_line
    line = result_line(impl="ours", value=123.0, ms=10.0, n_gpus=2, steps=5, warmup=3,
                       clocks={"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": []}, e2e_value=100.0, h2d=10, d2h=8,
                       gpu_launches=10, dtype="fp32", extra_config={"l2": "pool"})
    d = json.loads(line)
    assert "\n" not in line
    for k in ["metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "impl"]:
        assert k in d, k
    assert d["scaling"] == "strong" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["config"]["global_batch"] == 128 and d["config"]["parallelism"] == "dp2" and d["config"]["per_gpu_batch"] == 64
    assert set(d["e2e"]) == {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"}
    assert d["ms_per_step"] == 2.0


def test_reference_arm_reports_unavailable_or_runs_without_gpu():
    """On a box without CUDA the reference arm must print a single JSON line and exit 0."""
    import subprocess
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-500:]
    last = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")][-1]
    d = json.loads(last)
    assert d["impl"] == "reference" and ("unavailable" in d or "value" in d)


def test_pick_cluster_policy():
    from dist_tuto.pth_b200.ops.convnet_fused import pick_cluster
    assert [pick_cluster(b) for b in (128, 64, 32, 16, 8, 1)] == [1, 2, 4, 4, 8, 8]
    os.environ["B200DIST_CONVNET_CLUSTER"] = "1"
    try:
        assert pick_cluster(16) == 1
    finally:
        del os.environ["B200DIST_CONVNET_CLUSTER"]


def test_reference_copy_is_byte_identical():
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import install_ref
    ok, why = install_ref.verify()
    assert ok or "missing" in why, why
    # what the tests compare with (tests/golden/reference_convnet.npz) was recorded from the same bytes
    import numpy as np
    golden = np.load(os.path.join(ROOT, "tests", "golden", "reference_convnet.npz"))
    assert str(golden["train_dist_sha256"]) == json.load(open(install_ref.SHA_FILE))["train_dist.py"]


def test_aligned_start_gives_every_rank_the_same_instant():
    """The e2e window of both bench arms starts at a common instant (bench_common.aligned_start), gloo world 2 on the CPU."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import dist_tuto.pth_b200 as b2
    import dist_workers as W
    b2.launch(W.w_aligned_start, size=2, backend="gloo", join_timeout_s=120)
