"""The folded small-map route of layer3 / layer4 (frames as rows, UcFoldSlice in umma_conv.cuh) against the padded planar route
(LSD_FOLD=0).  Both multiply the same bf16 operands; the fold skips the taps that only read padding and sums in another fp32
order, so logits agree to a fraction of the bf16 budget and the layer3 output to within its stage bound.  The knob is read once
per process: each route runs in a fresh interpreter."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CODE = """
import sys; sys.path.insert(0, %r)
import json, numpy as np, torch, lipsync_b200 as lb
m = lb.LipSyncModel(); m.load_state_dict(lb.make_synthetic_state_dict(0)); m.to('cuda:0').eval(); m.compute_precision = 'bf16'
v, a = lb.synthetic_windows(41, 7)
out = {}
out['full'] = m(v.cuda(), a.cuda()).float().cpu().tolist()
out['half'] = m(v[:, :, 8:24].contiguous().cuda(), a[..., 32:96].contiguous().cuda()).float().cpu().tolist()
out['one'] = m(v[:3, :, :1].contiguous().cuda(), a[:3].cuda()).float().cpu().tolist()
v64, a64 = lb.synthetic_windows(43, 5, 32, 64, 64)
out['map64'] = m(v64.cuda(), a64.cuda()).float().cpu().tolist()
v2, a2 = lb.synthetic_windows(1, 2)
m(v2.cuda(), a2.cuda())
np.save(%r, m.planar_stage('y3', (2, 32, 6, 6, 256)).float().cpu().numpy())
print('OUT', json.dumps(out))
"""


def _run(env, y3_path):
    r = subprocess.run([sys.executable, "-c", CODE % (ROOT, y3_path)], env={**os.environ, **env}, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([l for l in r.stdout.splitlines() if l.startswith("OUT")][-1][4:]), np.load(y3_path)


def test_fold_matches_padded_route(tmp_path):
    fold, y3_fold = _run({}, str(tmp_path / "y3_fold.npy"))
    padded, y3_padded = _run({"LSD_FOLD": "0"}, str(tmp_path / "y3_padded.npy"))
    for k in ("full", "half", "one", "map64"):
        d = np.abs(np.asarray(fold[k]) - np.asarray(padded[k])).max()
        assert d <= 5e-3, (k, d, fold[k], padded[k])
    # layer3 output: the bound of the v_layer3 stage (relative to the stage's largest magnitude, tests/test_gpu_parity.py)
    rel = np.abs(y3_fold - y3_padded).max() / max(1e-12, float(np.abs(y3_padded).max()))
    assert rel <= 2e-2, rel
    assert np.abs(y3_padded).max() > 0
