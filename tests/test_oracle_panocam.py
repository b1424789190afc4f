"""CPU: the oracle's camera-parameters -> field restatement (oracle/panocam.py) against golden vectors produced by the
unmodified reference (tests/golden/panocam.npz, make_golden_panocam.py; reference_checks.npz, make_golden_reference_checks.py), and
the host-side closed form of general_vfov_to_focal against the reference's fsolve formulation."""
import ctypes
import os

import numpy as np
import pytest

from golden_util import from_byte_planes
from oracle import panocam as op

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "panocam.npz"))


def cases():
    return [tuple(c) for c in GOLD["cases"]]


@pytest.mark.parametrize("i", range(len(GOLD["cases"])))
def test_oracle_matches_reference_golden(i):
    f, w, h, el, roll, cx, cy = cases()[i]
    up = op.get_up_general(f, int(w), int(h), el, roll, cx, cy)
    lat = op.get_lat_general(f, int(w), int(h), el, roll, cx, cy)
    assert up.shape == (int(h), int(w), 2) and lat.shape == (int(h), int(w))
    assert np.abs(up - GOLD[f"up{i}"]).max() < 1e-12
    assert np.abs(lat - GOLD[f"lat{i}"]).max() < 1e-10
    assert np.allclose(np.linalg.norm(up, axis=2), 1.0, atol=1e-12)


def test_oracle_matches_live_reference():
    """Six random cameras (the reference's fields in tests/golden/reference_checks.npz)."""
    ref = np.load(os.path.join(os.path.dirname(__file__), "golden", "reference_checks.npz"))
    for i, (f, w, h, el, roll, cx, cy) in enumerate(ref["panocam/cases"]):
        w, h = int(w), int(h)
        up, lat = (from_byte_planes(ref[f"panocam/{n}{i}"], ref[f"panocam/{n}{i}/shape"]) for n in ("up", "lat"))
        assert np.abs(op.get_up_general(f, w, h, el, roll, cx, cy) - up).max() < 1e-12
        assert np.abs(op.get_lat_general(f, w, h, el, roll, cx, cy) - lat).max() < 1e-10


def test_closed_form_focal_matches_fsolve_formulation():
    from oracle.model import general_vfov_to_focal as ref          # utils/utils.py:47-91 restated with scipy.optimize.fsolve
    from perspectivefields_b200.panocam import general_vfov_to_focal
    rs = np.random.RandomState(0)
    cx, cy, g = rs.uniform(-0.3, 0.3, 64), rs.uniform(-0.3, 0.3, 64), rs.uniform(0.3, 2.2, 64)
    assert np.abs(general_vfov_to_focal(cx, cy, 1, g, False) - ref(cx, cy, 1, g, False)).max() < 1e-7   # fsolve stops at xtol = 1.5e-8
    assert abs(float(general_vfov_to_focal(0.0, 0.0, 1, 60.0, True)) - 0.5 / np.tan(np.radians(30.0))) < 1e-12


def test_pf_camera_struct_layout():
    from perspectivefields_b200 import _native
    assert ctypes.sizeof(_native.pf_camera) == 64          # include/pf_b200.h: 2 x int32, 5 x double, 2 x int64
    assert _native.pf_camera.up_offset.offset == 48 and _native.pf_camera.focal_rel.offset == 8
