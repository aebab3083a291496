"""ORACLE (test infrastructure): float64 restatement of branch attribution (`Predictor.branch_attribution`,
`lsd_branch_attribution`).

The head reads one 448-wide row per window, [cls 256 | raw 64 | delta 64 | hf 64].  f is the head in logit space: the artifact
fusion MLP of `lipsync_oracle.artifact_detector` (restated here, it is inline there) on the whole row, then
`lipsync_oracle.classifier` on cat[cls, fusion].  Players sync, raw, delta, hf are bits 0..3 of a coalition mask S; the hybrid
row x^{S,j} takes slice p from the window row when bit p is set and from background row b_j otherwise (the cls slice everywhere
the head reads cls).  v(S) = mean_j f(x^{S,j}), v(15) = f(x), phi_p = sum over S without p of w_|S| (v(S | p) - v(S)) with
w = (1/4, 1/12, 1/12, 1/4).
"""
from __future__ import annotations

from typing import Mapping

import numpy as np
import torch
import torch.nn.functional as F

from oracle import lipsync_oracle as orc

BRANCHES = ("sync", "raw", "delta", "hf")
SLICES = ((0, 256), (256, 320), (320, 384), (384, 448))
WEIGHTS = (1.0 / 4.0, 1.0 / 12.0, 1.0 / 12.0, 1.0 / 4.0)


def _f64(sd: Mapping[str, torch.Tensor]):
    return {k: v.double() for k, v in sd.items() if v.is_floating_point()}


def artifact_fusion(sd, comb: torch.Tensor) -> torch.Tensor:
    """artifact_detector.py's fusion MLP on cat[cls, raw, delta, hf] (as in `lipsync_oracle.artifact_detector`)."""
    p = "artifact_detector.artifact_fusion"
    h = F.relu(comb @ sd[p + ".0.weight"].t() + sd[p + ".0.bias"])
    return F.relu(h @ sd[p + ".2.weight"].t() + sd[p + ".2.bias"])


def head(sd, x) -> np.ndarray:
    """f: (N, 448) head input rows -> (N,) float64 logits."""
    sd = _f64(sd)
    x = torch.as_tensor(np.asarray(x, dtype=np.float64))
    return orc.classifier(sd, torch.cat([x[:, :256], artifact_fusion(sd, x)], dim=-1)).numpy()


def hybrid(x, b, S: int) -> np.ndarray:
    """x^{S}: slice p from row x when bit p of S is set, from row b otherwise."""
    out = np.array(b, dtype=np.float64, copy=True)
    for p, (lo, hi) in enumerate(SLICES):
        if (S >> p) & 1:
            out[..., lo:hi] = np.asarray(x, dtype=np.float64)[..., lo:hi]
    return out


def coalition_values(sd, feats, background) -> np.ndarray:
    """(n, 448) windows, (M, 448) background -> (n, 16) float64 v_i(S)."""
    x = np.asarray(feats, dtype=np.float64)
    bg = np.asarray(background, dtype=np.float64)
    n, M = x.shape[0], bg.shape[0]
    v = np.zeros((n, 16))
    for S in range(15):
        rows = hybrid(x[:, None, :], np.broadcast_to(bg[None], (n, M, bg.shape[1])), S).reshape(n * M, -1)
        v[:, S] = head(sd, rows).reshape(n, M).mean(axis=1)
    v[:, 15] = head(sd, x)
    return v


def shapley(values) -> np.ndarray:
    """(n, 16) coalition values of 4-player games -> (n, 4) Shapley values."""
    v = np.asarray(values, dtype=np.float64).reshape(-1, 16)
    phi = np.zeros((v.shape[0], 4))
    for p in range(4):
        for S in range(16):
            if not (S >> p) & 1:
                phi[:, p] += WEIGHTS[bin(S).count("1")] * (v[:, S | (1 << p)] - v[:, S])
    return phi
