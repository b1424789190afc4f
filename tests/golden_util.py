"""Helpers shared by the golden-fixture tests (oracle on CPU, CUDA path on the GPU box)."""
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def manifest():
    with open(os.path.join(GOLDEN_DIR, "manifest.json")) as f:
        return json.load(f)


def load_golden(version):
    m = manifest()
    return m, dict(np.load(os.path.join(GOLDEN_DIR, m["versions"][version]["file"])))


def golden_images():
    from oracle import weights_gen as wg

    m = manifest()
    return wg.synth_images(1, 480, 640, m["seed"]) + wg.smooth_images(1, 360, 500, m["seed"])


def rel_err(a, b):
    """max|a-b| / max|b|  -- the 'relative fp32 tolerance' metric of BASELINE.md (b = reference)."""
    a = torch.as_tensor(a, dtype=torch.float64)
    b = torch.as_tensor(b, dtype=torch.float64)
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def byte_planes(a):
    """A float64 array as its 8 byte planes (uint8 [8, numel]): smooth fields stored this way compress about 20 % better."""
    return np.ascontiguousarray(a, np.float64).view(np.uint8).reshape(-1, 8).T.copy()


def from_byte_planes(p, shape):
    return np.ascontiguousarray(p.T).view(np.float64).reshape(tuple(shape))


def compare_with_golden(version, results, tol, check_stats=True, skip_keys=()):
    """Compare a list of result dicts (one per golden image) with the stored reference outputs.
    Returns {key: worst relative error}."""
    m, g = load_golden(version)
    worst = {}
    for i, res in enumerate(results):
        w = compare_result(res, g, f"{i}/", m["versions"][version]["keys"][i], m["stride"], m["logit_stride"], tol,
                           f"{version} img{i}", check_stats, skip_keys)
        for k, e in w.items():
            worst[k] = max(worst.get(k, 0.0), e)
    return worst


def subsample(v, stride, logit_stride, edges=False):
    """The rows and columns of ``v`` (torch, [..., H, W]) at ``stride`` (``logit_stride`` for logit tensors); ``edges`` adds
    the last row and column when the stride misses them."""
    if v.ndim < 2:
        return v
    st = logit_stride if (v.ndim == 3 and v.shape[0] > 3) else stride

    def index(n):
        i = list(range(0, n, st))
        return i + [n - 1] if edges and i[-1] != n - 1 else i
    return v[..., index(v.shape[-2]), :][..., index(v.shape[-1])]


def compare_result(res, g, prefix, keys, stride, logit_stride, tol, label, check_stats=True, skip_keys=(), edges=False):
    """Compare one result dict with reference outputs stored under ``prefix`` in ``g``: each tensor as a sub-sample
    (``subsample``) plus its float64 (sum, abs-sum, numel).  Returns {key: relative error}."""
    assert list(res.keys()) == list(keys), (list(res.keys()), list(keys))
    worst = {}
    for k, v in res.items():
        if isinstance(v, str):
            assert v == "deg"
            continue
        if k in skip_keys:
            continue
        v = v.detach().cpu().float()
        assert tuple(v.shape) == tuple(g[f"{prefix}{k}/shape"]), (k, v.shape)
        e = rel_err(subsample(v, stride, logit_stride, edges), g[f"{prefix}{k}"])
        worst[k] = e
        assert e <= tol, f"{label} {k}: rel err {e:.3g} > {tol}"
        if check_stats:
            s, sa, n = g[f"{prefix}{k}/stats"]
            assert abs(v.double().abs().sum().item() - sa) <= tol * max(sa, 1e-30) * 4, (k, "abs-sum checksum")
    return worst
