"""Pins oracle/dit.py (and, on the GPU, the CUDA denoiser itself) to the REFERENCE'S OWN denoiser code.

tests/golden/make_dit_golden.py executes the reference's DGSDenoiser classes from diffusionGS/models/denoiser/denoiser.py
and denoiser_scene.py -- with DiTBlock / modulate from models/transformers/utils_transformer.py -- by path
(tests/golden/ref_import.py; only absent third-party packages are stubbed) and stores what they produce:
* tests/golden/dit_ref_pins.npz: the reference's parameter names and shapes, gradient norms and sketches, and the outputs
  of its building blocks; oracle/dit.py must equal them to 1e-6 relative (outputs) and 2e-5 (parameter gradients);
* tests/golden/dit_ref_*.npz: the outputs of every case; the oracle must reproduce them, and on a GPU the product's
  dgs_dit_forward must match them within the north-star bound for bf16 (1e-3 relative, norm-wise).
"""
import hashlib
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_dit_golden as mdg  # noqa: E402
import ref_import as ri  # noqa: E402

from oracle.dit import DenoiserOracle  # noqa: E402

SMALL = [n for n in ri.DIT_CASES if n.startswith("s_")]
WIDE = [n for n in ri.DIT_CASES if n.startswith("w1024_")]


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float(((a - b).norm() / (b.norm() + 1e-30)).detach())


def _oracle_for(name):
    scene, pe, cfg, _, seed = ri.DIT_CASES[name]
    o = DenoiserOracle(width=cfg["width"], heads=cfg["width"] // cfg["dim_heads"], layers=cfg["num_layers"],
                       patch=cfg["patch_size"], scene=scene, ray_pe_type=pe)
    o.load_state_dict(ri.seeded_state_dict(o, seed), strict=True)
    return o


def _fixture(name):
    z = np.load(os.path.join(HERE, "golden", f"dit_ref_{name}.npz"))
    return {k[4:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("out/")}, z


@pytest.mark.parametrize("name", mdg.PINNED)
def test_oracle_equals_reference_code(name):
    torch.manual_seed(0)
    _, _, _, (b, v, h, w), seed = ri.DIT_CASES[name]
    pins = np.load(mdg.PINS)
    o = _oracle_for(name)
    # identical module tree: the reference's parameters, seeded in its own order, load strictly (same keys and shapes)
    o.load_state_dict(ri.seeded_params(mdg.shapes(pins, name), seed), strict=True)
    img, ro, rd, t = ri.seeded_dit_inputs(b, v, h, w, seed + 1000)
    oo, oia = o.image_to_gaussians(img, ro, rd, t)
    oo = dict(oo, img_aligned_xyz=oia)
    outs, _ = _fixture(name)
    for k in outs:
        e = rel(oo[k].detach(), outs[k])
        assert e < 1e-6, (name, k, e)
    cot = {k: ri.seeded(tuple(oo[k].shape), seed + 2000 + i) for i, k in enumerate(ri.GS_KEYS)}
    loss = sum((oo[k] * cot[k]).sum() for k in cot)
    og = torch.autograd.grad(loss, list(o.parameters()))
    ref = mdg.gradient_digests(pins, name)
    worst = max(ri.sketched_rel(g, *ref[k]) for (k, _), g in zip(o.named_parameters(), og))
    assert worst < 2e-5, (name, worst)  # fp32 autograd through SDPA vs explicit softmax: summation order only


def test_reference_blocks_one_by_one():
    """TimestepEmbedder, DiTBlock, GaussiansUpsampler, ImageTokenDecoder of the reference, each against its restatement."""
    from oracle import dit as od
    pins = np.load(mdg.PINS)
    D, H = mdg.BLOCK_WIDTH, mdg.BLOCK_HEADS
    x, c, t = mdg.block_inputs()
    mine = {"DiTBlock": (od.DiTBlock(D, H), (x, c)), "TimestepEmbedder": (od.TimestepEmbedder(D), (t,)),
            "GaussiansUpsampler": (od._Head(D, 14), (x, c)), "ImageTokenDecoder": (od._Head(D, 16 * 14), (x, c))}
    for name, (m, args) in mine.items():
        m.load_state_dict(ri.seeded_params(mdg.shapes(pins, "blocks/" + name), 5), strict=True)
        assert rel(m(*args), torch.from_numpy(pins[f"blocks/{name}/out"])) < 1e-6, name
    # bit-exact: the digest of the reference's modulate() output
    assert hashlib.sha256(od.modulate(x, c, 2 * c).numpy().tobytes()).hexdigest() == str(pins["blocks/modulate_sha256"])


def test_oracle_attention_equals_sdpa():
    from oracle.dit import Attention
    torch.manual_seed(1)
    a = Attention(128, 4)
    x = torch.randn(2, 50, 128)
    B, N, C = x.shape
    q, k, v = a.qkv(x).reshape(B, N, 3, 4, 32).permute(2, 0, 3, 1, 4).unbind(0)
    ref = a.proj(torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(B, N, C))
    assert rel(a(x), ref) < 1e-6


@pytest.mark.parametrize("name", SMALL + WIDE)
def test_oracle_reproduces_committed_reference_outputs(name):
    if name.startswith("w1024") and os.environ.get("DGS_SKIP_WIDE_CPU"):
        pytest.skip("wide cases skipped by request")
    _, _, _, (b, v, h, w), seed = ri.DIT_CASES[name]
    gold, z = _fixture(name)
    o = _oracle_for(name)
    img, ro, rd, t = ri.seeded_dit_inputs(b, v, h, w, seed + 1000)
    oo, oia = o.image_to_gaussians(img, ro, rd, t)
    oo = dict(oo, img_aligned_xyz=oia)
    for k, g in gold.items():
        assert rel(oo[k].detach(), g) < 1e-5, (name, k)  # BLAS summation order may differ between boxes
    if name.startswith("s_"):
        cot = {k: ri.seeded(tuple(oo[k].shape), seed + 2000 + i) for i, k in enumerate(ri.GS_KEYS)}
        loss = sum((oo[k] * cot[k]).sum() for k in cot)
        og = torch.autograd.grad(loss, list(o.parameters()))
        rng = np.random.default_rng(7)
        for (k, _), g in zip(o.named_parameters(), og):
            gg = g.double().numpy().ravel()
            n_ref, p_ref = float(z["gnorm/" + k]), float(z["gproj/" + k])
            proj = float(gg @ rng.standard_normal(gg.size))
            assert abs(np.linalg.norm(gg) - n_ref) <= 1e-4 * n_ref + 1e-12, (name, k)
            assert abs(proj - p_ref) <= 1e-3 * n_ref + 1e-9, (name, k)  # the projection has standard deviation ~ |g|


@pytest.mark.gpu
@pytest.mark.parametrize("name", WIDE)
def test_cuda_denoiser_matches_reference_outputs(name):
    """The product (dgs_dit_forward through DGSDenoiser[Scene]) against numbers the reference's own code produced."""
    from dgs_b200.denoiser import DGSDenoiser, DGSDenoiserScene
    scene, pe, cfg, (b, v, h, w), seed = ri.DIT_CASES[name]
    model = (DGSDenoiserScene if scene else DGSDenoiser)(dict(cfg, in_channels=9, n_gaussians=2, ray_pe_type=pe))
    model.load_state_dict(ri.seeded_state_dict(model, seed), strict=True)
    model = model.to("cuda:0")
    img, ro, rd, t = [a.to("cuda:0") for a in ri.seeded_dit_inputs(b, v, h, w, seed + 1000)]
    out, ia = model.image_to_gaussians(img, ro, rd, t)
    torch.cuda.synchronize()
    gold, _ = _fixture(name)
    got = dict(out, img_aligned_xyz=ia)
    for k, g in gold.items():
        e = rel(got[k].cpu(), g)
        print(f"{name} {k}: rel={e:.2e}")
        assert e < 1e-3, (name, k, e)  # north-star bound for bf16 operands
