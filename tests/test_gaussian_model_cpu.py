"""GaussianModel post-processing after the sampler loop (SURVEY 8f row 3): filters against what the REFERENCE's own
GaussianModel (gs_core.py:386-475, executed by path in tests/golden/make_renderer_golden.py) kept, and the PLY export
(gs_core.py:577-713) by parsing the written file."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_renderer_golden as mg  # noqa: E402

from dgs_b200.renderer import GaussianModel  # noqa: E402


def test_filters_equal_reference_gaussian_model():
    ref = np.load(mg.GAUSSIAN_MODEL)
    ours = GaussianModel(0).set_data(*mg.gaussian_data())
    ours.apply_all_filters(**mg.FILTERS)
    assert 0 < ours._xyz.shape[0] < 500
    for k in mg.GAUSSIAN_MODEL_FIELDS:
        assert torch.equal(getattr(ours, k), torch.from_numpy(ref[k])), k
    assert ours.construct_dtypes() == [tuple(e.split(":")) for e in ref["dtypes"]]


def test_save_ply_layout(tmp_path):
    m = GaussianModel(0).set_data(*mg.gaussian_data(37, seed=3))
    path = m.save_ply(str(tmp_path / "sub" / "g.ply"))
    raw = open(path, "rb").read()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode().strip().split("\n")
    assert lines[:3] == ["ply", "format binary_little_endian 1.0", "element vertex 37"]
    props = [l.split()[1:] for l in lines[3:]]
    names = [p[1] for p in props]
    assert names[:9] == ["x", "y", "z", "red", "green", "blue", "f_dc_0", "f_dc_1", "f_dc_2"]
    assert names[9:9 + 45] == [f"f_rest_{i}" for i in range(45)]           # padded to SH degree 3 for the viewers
    assert names[-8:] == ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"]
    dt = np.dtype([(n, "<f4" if t == "float" else "u1") for t, n in props])
    el = np.frombuffer(body, dtype=dt)
    assert el.shape == (37,)
    assert np.allclose(np.stack([el["x"], el["y"], el["z"]], 1), m._xyz.numpy())
    assert np.allclose(el["opacity"], m._opacity.numpy()[:, 0]) and np.allclose(el["rot_3"], m._rotation.numpy()[:, 3])
    rgb = ((m._features_dc[:, 0].numpy() * 0.28209479177387814 + 0.5) * 255).clip(0, 255).astype(np.uint8)
    assert np.array_equal(np.stack([el["red"], el["green"], el["blue"]], 1), rgb)
    assert float(np.abs(el["f_rest_0"]).max()) == 0.0
