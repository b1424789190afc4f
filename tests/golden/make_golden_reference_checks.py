"""Generate tests/golden/reference_checks.npz and tests/golden/reference_config.json.gz from the UNMODIFIED reference:

    python tests/golden/make_golden_reference_checks.py      # needs the reference checkout (oracle/ref_shim.py)

They hold what tests/test_oracle_vs_reference.py and tests/test_oracle_panocam.py compare the oracle with, so that those
tests run without the reference:

* reference_config.json.gz: per zoo version, the reference model's state-dict keys and shapes in order, its merged yacs
  configuration and its ``model_zoo`` entry.
* reference_checks.npz: ``inference_batch`` of PersNet_Paramnet-GSV-uncentered (synthetic checkpoint seed 3, one smooth
  300x420 image, seed 5) under ``live/``; the float-input branch of Paramnet-360Cities-edina-centered (seed 0, smooth 200x260
  image, seed 9, as float32 + 0.25) under ``float/``, with the shape and SHA-256 of ``aug.apply_image``'s output under
  ``float/resized``; ``PanoCam`` up-vector / latitude fields for six random cameras under ``panocam/``, whole (as byte
  planes, tests/golden_util.py:byte_planes).  The model outputs are stored as the rows and columns at ``stride`` plus the
  last row and column (tests/golden_util.py:subsample) with float64 checksums of the whole tensor, as
  tests/golden/make_golden.py does.
"""
import gzip
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from golden_util import byte_planes, subsample  # noqa: E402
from oracle import weights_gen as wg  # noqa: E402
from oracle.ref_shim import load_reference  # noqa: E402
from oracle.variants import VARIANTS  # noqa: E402

STRIDE = 8
LOGIT_STRIDE = 16
OUT = os.path.join(ROOT, "tests", "golden")


def store_result(arrays, prefix, res):
    arrays[prefix + "keys"] = np.array(list(res.keys()))
    for k, v in res.items():
        if isinstance(v, str):
            continue
        arrays[prefix + k] = subsample(v.detach().cpu().float(), STRIDE, LOGIT_STRIDE, edges=True).numpy()
        v64 = v.detach().double()
        arrays[prefix + k + "/stats"] = np.array([v64.sum().item(), v64.abs().sum().item(), v64.numel()], np.float64)
        arrays[prefix + k + "/shape"] = np.array(v.shape, np.int64)


def write_checkpoint(th, version, sd):
    torch.save({"model": sd}, os.path.join(th, "hub", "checkpoints", VARIANTS[version]["ckpt"]))


def to_json(x):
    if isinstance(x, dict):
        return {k: to_json(v) for k, v in x.items()}
    if isinstance(x, (list, tuple)):
        return [to_json(v) for v in x]
    return x


def main():
    th = tempfile.mkdtemp(prefix="pf_golden_")
    os.environ["TORCH_HOME"] = th
    os.makedirs(os.path.join(th, "hub", "checkpoints"), exist_ok=True)
    p2d = load_reference()
    from oracle.schema import state_dict_schema

    config = {"schema": {}, "cfg": {}, "model_zoo": {}}
    for version in VARIANTS:
        write_checkpoint(th, version, {k: torch.zeros(s) for k, s in state_dict_schema(version)})
        model = p2d.PerspectiveFields(version)
        config["schema"][version] = [[k, list(v.shape)] for k, v in model.state_dict().items()]
        config["cfg"][version] = to_json(model.cfg)
        config["model_zoo"][version] = p2d.perspectivefields.model_zoo[version]
    with gzip.GzipFile(os.path.join(OUT, "reference_config.json.gz"), "wb", mtime=0) as f:
        f.write(json.dumps(config, indent=0, sort_keys=False).encode())

    arrays = {"stride": np.array(STRIDE), "logit_stride": np.array(LOGIT_STRIDE), "edges": np.array(True)}
    version = "PersNet_Paramnet-GSV-uncentered"
    sd = wg.synth_state_dict(version, 3)
    write_checkpoint(th, version, sd)
    store_result(arrays, "live/", p2d.PerspectiveFields(version).eval().inference_batch(wg.smooth_images(1, 300, 420, 5))[0])

    version = "Paramnet-360Cities-edina-centered"
    sd = wg.synth_state_dict(version, 0)
    write_checkpoint(th, version, sd)
    model = p2d.PerspectiveFields(version).eval()
    img = wg.smooth_images(1, 200, 260, 9)[0].astype(np.float32) + 0.25
    resized = model.aug.apply_image(img)
    arrays["float/resized/shape"] = np.array(resized.shape, np.int64)
    arrays["float/resized/sha256"] = np.array(hashlib.sha256(np.ascontiguousarray(resized).tobytes()).hexdigest())
    store_result(arrays, "float/", model.inference(img))

    from perspective2d.utils.panocam import PanoCam
    rs = np.random.RandomState(3)
    cases = []
    for i in range(6):
        f, el, roll = rs.uniform(0.3, 2.0), rs.uniform(-1.4, 1.4), rs.uniform(-3.1, 3.1)
        cx, cy = rs.uniform(-0.3, 0.3, 2)
        w, h = int(rs.randint(2, 60)), int(rs.randint(2, 60))
        cases.append((f, w, h, el, roll, cx, cy))
        for name, field in (("up", PanoCam.get_up_general(f, w, h, el, roll, cx, cy)),
                            ("lat", PanoCam.get_lat_general(f, w, h, el, roll, cx, cy))):
            arrays[f"panocam/{name}{i}"] = byte_planes(field)
            arrays[f"panocam/{name}{i}/shape"] = np.array(field.shape, np.int64)
    arrays["panocam/cases"] = np.array(cases, np.float64)
    path = os.path.join(OUT, "reference_checks.npz")
    np.savez_compressed(path, **arrays)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
