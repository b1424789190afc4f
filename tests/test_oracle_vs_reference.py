"""CPU: the oracle against what the unmodified reference computed for the same inputs, stored under tests/golden/ by
tests/golden/make_golden_reference_checks.py: its state-dict layout, merged configuration and model-zoo entry per version
(reference_config.json.gz), and its outputs on seeded synthetic checkpoints and images (reference_checks.npz)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from golden_util import GOLDEN_DIR, compare_result
from oracle import model as om
from oracle import weights_gen as wg
from oracle.schema import state_dict_schema
from oracle.variants import VARIANTS

with gzip.open(os.path.join(GOLDEN_DIR, "reference_config.json.gz"), "rt") as _f:
    REF_CONFIG = json.load(_f)
REF = np.load(os.path.join(GOLDEN_DIR, "reference_checks.npz"))


def _compare(res, prefix, label):
    compare_result(res, REF, prefix, REF[prefix + "keys"].tolist(), int(REF["stride"]), int(REF["logit_stride"]), 1e-4, label,
                   edges=bool(REF["edges"]))


@pytest.mark.parametrize("version", list(VARIANTS))
def test_schema_matches_reference(version):
    ref = REF_CONFIG["schema"][version]
    assert [k for k, _ in ref] == [k for k, _ in state_dict_schema(version)]
    for (k, s), (_, rs) in zip(state_dict_schema(version), ref):
        assert tuple(rs) == tuple(s), k


def test_live_outputs_match():
    version = "PersNet_Paramnet-GSV-uncentered"
    sd = wg.synth_state_dict(version, 3)
    imgs = wg.smooth_images(1, 300, 420, 5)
    ora = om.inference_batch(sd, version, imgs)
    _compare(ora[0], "live/", version)


def test_float_input_branch_matches_reference():
    """perspectivefields.py:47-66: non-uint8 images go through F.interpolate instead of PIL (pins oracle.model.inference_float /
    resize_float, which tests/test_gpu_forward.py uses as the referee for the CUDA float branch)."""
    version = "Paramnet-360Cities-edina-centered"
    sd = wg.synth_state_dict(version, 0)
    img = wg.smooth_images(1, 200, 260, 9)[0].astype(np.float32) + 0.25
    resized = om.resize_float(img, 320, 320)
    assert resized.shape == tuple(REF["float/resized/shape"]) and resized.dtype == np.float32
    assert hashlib.sha256(np.ascontiguousarray(resized).tobytes()).hexdigest() == str(REF["float/resized/sha256"])
    _compare(om.inference_float(sd, version, img), "float/", version)


def test_yaml_configuration_matches_reference():
    """perspectivefields_b200/config/*.yaml (defaults + per-variant overrides, parsed with PyYAML) give every inference-relevant
    field the value the reference's yacs tree has after merge_from_file (perspectivefields.py:124-131)."""
    from perspectivefields_b200 import variants as V

    for version in VARIANTS:
        ref = REF_CONFIG["cfg"][version]
        mine = V.make_cfg(version)

        def walk(a, b, path):
            for k, v in a.items():
                assert k in b, (version, path + k)
                if isinstance(v, dict):
                    walk(v, b[k], path + k + ".")
                else:
                    rv = b[k]
                    rv = list(rv) if isinstance(rv, (list, tuple)) else rv
                    assert rv == v, (version, path + k, rv, v)
        walk(mine, ref, "")
        assert V.model_zoo[version] == REF_CONFIG["model_zoo"][version]
