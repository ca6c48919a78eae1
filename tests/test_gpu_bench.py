"""bench.py --dump-outputs: what the last timed step returned, identical for two runs with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "3",
                        "--warmup", "1", "--no-cpu-baseline", "--no-kernel-times", "--no-aux-workload",
                        "--dump-outputs", str(out_dir), *extra], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


@pytest.mark.parametrize("extra", [(), ("--bi-graphs", "dense"), ("--with-aux",)])
def test_dump_outputs_of_the_last_timed_step(tmp_path, extra):
    res, a = _run(tmp_path / "a", *extra)
    n_cats, c_uni, B, h, w = [5, 3, 7], 11, 4, 16, 32  # bench.WORKLOADS["tiny"]
    want = {"loss", "miou", "confusion", "dlogits_uni"}
    if "dense" in extra:
        want |= {f"dbi_graph{d}" for d in range(3)}
    if "--with-aux" in extra:
        want |= {f"daux{d}" for d in range(3)}
    assert set(a) == want and all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert res["steps"] == 3
    assert float(a["loss"]) == res["loss"]  # the JSON line reports the loss of the last timed step
    assert a["confusion"].dtype == np.float64 and a["confusion"].shape == (sum(c * c for c in n_cats),)
    assert a["confusion"].sum() == res["hist_check"]["hist_sum"]
    assert a["miou"].shape == (3,) and a["dlogits_uni"].shape == (B, c_uni, h, w)
    assert np.isfinite(a["dlogits_uni"]).all() and np.abs(a["dlogits_uni"]).max() > 0
    for d, c in enumerate(n_cats):
        if "dense" in extra:
            assert a[f"dbi_graph{d}"].shape == (c, c_uni)
        if "--with-aux" in extra:
            assert a[f"daux{d}"].shape == (B, c, h, w)
    if not extra:  # the same arguments give the same inputs, so a second run reproduces every output
        _, b = _run(tmp_path / "b")
        assert set(b) == want
        for k in want:
            np.testing.assert_allclose(a[k], b[k], rtol=1e-6, atol=1e-9, err_msg=k)
