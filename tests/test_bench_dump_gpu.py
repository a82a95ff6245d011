"""GPU: ``bench.py --dump-outputs`` writes what the last timed step handed its caller, as float32 .npy files, and
``--steps`` sets the number of timed steps; run at a tiny shape."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, V, N, L = 4, 12, 16, 24


def _bench(mode, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--mode", mode,
                        "--batch", str(B), "--views", str(V), "--nodes", str(N), "--tokens", str(L), "--x-layers", "1",
                        "--no-soak", "--no-cpu-baseline", "--no-gpu-eager", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.strip()][-1])
    assert line["steps"] == 3
    arrays = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
    assert all(x.dtype == np.float32 for x in arrays.values())
    return arrays


@pytest.mark.parametrize("mode", ["fwd", "train"])
def test_dump_outputs(mode, tmp_path):
    d = _bench(mode, tmp_path)
    want = {"global_logits": (B, N), "global_logits_masked": (B, N)}
    if mode == "fwd":
        want.update(pano_embeds=(B, V, 768), pano_masks=(B, V), gmap_embeds=(B, N, 768))
    else:
        want["params"] = d["params"].shape
        assert d["params"].ndim == 1
    assert {k: v.shape for k, v in d.items()} == want
    assert all(np.isfinite(x).all() for x in d.values())
    m = d["global_logits_masked"]
    assert set(np.unique(m)) <= {0.0, 1.0} and (m == 0).any(axis=1).all() and (m == 1).any()
    assert (d["global_logits"][m == 1] == 0).all()
