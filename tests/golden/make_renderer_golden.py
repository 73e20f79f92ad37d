"""Writes tests/golden/renderer_ref_<case>.npz: the REFERENCE's own Python renderer stack --
diffusionGS/models/gsrenderer/renderer.py (Renderer.forward), gs_core.py (Camera, GaussianModel activations,
render_opencv_cam, DeferredGaussianRender.forward/backward) and the diff_gaussian_rasterization binding classes --
executed by path from /root/reference on CPU tensors.  Only the compiled `_C` extension underneath is replaced, by the CPU
oracle (oracle/raster.py, itself held to the reference's CUDA kernels by tests/golden/ref_*.npz).  Stored: the seeded
inputs, the rendered views and the five parameter gradients of a seeded cotangent.

Also writes tests/golden/gaussian_model_ref.npz: what the reference's GaussianModel (gs_core.py:386-475, 578-633) keeps
after apply_all_filters on seeded Gaussians, and the PLY property list it builds.

    python tests/golden/make_renderer_golden.py        # needs /root/reference (this container)
"""
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [HERE, ROOT, os.path.join(ROOT, "open-diffusiongs_b200")]
import ref_import as ri  # noqa: E402
from dgs_b200 import synth  # noqa: E402

NAMES = ("xyz", "features", "scaling", "rotation", "opacity")
# name -> (B, V, P, W, H, distribution, seed)
CASES = {"trained_b2v3": (2, 3, 1500, 64, 48, "trained", 0), "init_b1v2": (1, 2, 800, 48, 48, "init", 5),
         "fine_b1v4": (1, 4, 3000, 80, 64, "fine", 9)}
GAUSSIAN_MODEL = os.path.join(HERE, "gaussian_model_ref.npz")
GAUSSIAN_MODEL_FIELDS = ("_xyz", "_features_dc", "_scaling", "_rotation", "_opacity")
FILTERS = dict(opacity_thres=0.05, crop_bbx=[-1, 1, -1, 1, -1, 1],
               cam_origins=torch.tensor([[0.0, 0.0, 3.0], [3.0, 0.0, 0.0], [0.0, 3.0, 1.0]]), nearfar_percent=(0.005, 1.0))


def inputs(case):
    B, V, P, W, H, dist, seed = CASES[case]
    gs = [synth.make_gaussians(P, seed + i, dist) for i in range(B)]
    raw = {k: np.stack([g[k] for g in gs]) for k in NAMES}
    rng = np.random.default_rng(seed + 100)
    raw["rotation"] = raw["rotation"] * rng.uniform(0.5, 2.0, (B, P, 1)).astype(np.float32)  # un-normalised on purpose
    cams = [synth.orbit_cameras(V, W, H, az0=15.0 * i + seed) for i in range(B)]
    c2w, fx = np.stack([c[0] for c in cams]), np.stack([c[1] for c in cams])
    fx[..., 2] += rng.uniform(-2, 2, fx.shape[:-1]).astype(np.float32)  # off-centre principal points
    fx[..., 3] += rng.uniform(-2, 2, fx.shape[:-1]).astype(np.float32)
    dimg = rng.normal(0, 1, (B, V, 3, H, W)).astype(np.float16).astype(np.float32)  # stored as fp16, exactly
    return raw, c2w.astype(np.float32), fx.astype(np.float32), dimg, H, W


def run_reference(case):
    ns = ri.load("oracle")
    raw, c2w, fx, dimg, H, W = inputs(case)
    renderer = ns.renderer.Renderer(SimpleNamespace(gaussians_sh_degree=0, use_gssplat=False))
    params = [torch.tensor(raw[k], requires_grad=True) for k in NAMES]
    with ri.cpu_device_shim():
        img = renderer(*params, H, W, torch.tensor(c2w), torch.tensor(fx))
        img.backward(torch.tensor(dimg))
    return raw, c2w, fx, dimg, img.detach().numpy(), {k: p.grad.numpy() for k, p in zip(NAMES, params)}


def gaussian_data(n=500, seed=0):
    """(xyz, features, scaling, rotation, opacity) of n seeded Gaussians, SH degree 0"""
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(n, 3, generator=g) * 0.8, torch.randn(n, 1, 3, generator=g), torch.randn(n, 3, generator=g) - 3,
            torch.randn(n, 4, generator=g), torch.randn(n, 1, generator=g) * 2)


def write_gaussian_model():
    ref = ri.load("oracle").gs_core.GaussianModel(0).set_data(*gaussian_data())
    ref.apply_all_filters(**FILTERS)
    rec = {k: getattr(ref, k).numpy() for k in GAUSSIAN_MODEL_FIELDS}
    rec["dtypes"] = np.array([f"{n}:{t}" for n, t in ref.construct_dtypes()])
    np.savez_compressed(GAUSSIAN_MODEL, **rec)
    print(GAUSSIAN_MODEL, os.path.getsize(GAUSSIAN_MODEL), "bytes")


def main():
    write_gaussian_model()
    for case in CASES:
        raw, c2w, fx, dimg, img, grads = run_reference(case)
        rec = {"in/" + k: v for k, v in raw.items()}
        rec.update({"in/c2w": c2w, "in/fxfycxcy": fx, "in/dimg": dimg.astype(np.float16), "out/img": img})
        rec.update({"grad/" + k: v for k, v in grads.items()})
        path = os.path.join(HERE, f"renderer_ref_{case}.npz")
        np.savez_compressed(path, **rec)
        print(case, img.shape, f"mean={img.mean():.4f}", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
