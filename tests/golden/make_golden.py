"""Generates tests/golden/ref_*.npz by running the UNMODIFIED reference kernels (oracle/_ref/dgr_ref_C.so,
built by oracle/build_ref.py from /root/reference) on a B200, on the seeded C1 scenes of tests/util.py.
Run on the GPU box:   python tests/golden/make_golden.py gpurun_out/golden
then copy gpurun_out/golden/*.npz to tests/golden/ and commit them.  Stored fp16-free, fp32 arrays,
small scenes so the fixtures stay < 1 MB each.

Also writes ref_noise_floors.json: on each case of precomp_cases(), the rel-L2 of the reference kernels' fp32 gradients
against the fp64-accumulating CPU oracle -- the atomics-order / cancellation noise of the specification itself, which
tests/test_raster_gpu.py allows our kernels twice of."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "open-diffusiongs_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

from oracle import build_ref  # noqa: E402
from util import oracle_forward, rel_l2, scene_c1  # noqa: E402

CASES = [  # (name, P, dist, W, H, seed, degree)
    ("trained_2k_128", 2000, "trained", 128, 128, 0, 0),
    ("init_1k_96x64", 1000, "init", 96, 64, 1, 0),
    ("fine_4k_128", 4000, "fine", 128, 128, 2, 0),
    ("trained_1k_sh2", 1000, "trained", 64, 64, 3, 2),
]
NOISE_FLOORS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "ref_noise_floors.json")
GRAD_NAMES = ["dL_dmeans2D", "dL_dcolors", "dL_dopacity", "dL_dmeans3D", "dL_dcov3D", "dL_dsh", "dL_dscales", "dL_drotations"]


def precomp_cases():
    """-> (scene, dL/dpix, {tag: forward keyword arguments}): SH degrees 1-3, precomputed colours, precomputed 3D
    covariances on one 3000-Gaussian scene."""
    sc = scene_c1(P=3000, dist="trained", W=160, H=96)
    rng = np.random.default_rng(7)
    dpix = rng.normal(0, 1, (3, sc["H"], sc["W"])).astype(np.float32)
    sh = rng.normal(0, 0.4, (sc["P"], 16, 3)).astype(np.float32)
    cases = {f"sh{deg}": dict(sh=sh, degree=deg) for deg in (1, 2, 3)}
    cases["colors_precomp"] = dict(colors=rng.uniform(0, 1, (sc["P"], 3)).astype(np.float32))
    cases["cov_precomp"] = dict(cov3d=oracle_forward(sc)["cov3D"])
    return sc, dpix, cases


def write_noise_floors(ref, path):
    from oracle import raster as orc
    dev = "cuda:0"
    T = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float32, device=dev)  # noqa: E731
    e = torch.empty(0, device=dev)
    sc, dpix, cases = precomp_cases()
    a = sc["act"]
    floors = {}
    for tag, kw in cases.items():
        colors, cov3d, deg = kw.get("colors"), kw.get("cov3d"), kw.get("degree", 0)
        col = e if colors is None else T(colors)
        cov = e if cov3d is None else T(cov3d)
        args = (T(np.ones(3)), T(a["means3D"]), col, T(a["opacities"]), e if cov3d is not None else T(a["scales"]),
                e if cov3d is not None else T(a["rotations"]), 1.0, cov, T(sc["view"]), T(sc["proj"]), float(sc["tanx"]),
                float(sc["tany"]), sc["H"], sc["W"], e if colors is not None else T(kw.get("sh", a["shs"])), deg,
                T(sc["campos"]), False, False)
        R, _, radii, geom, binning, img = ref.rasterize_gaussians(*args)
        g = ref.rasterize_gaussians_backward(args[0], args[1], radii, col, args[4], args[5], 1.0, cov, args[8], args[9],
                                             args[10], args[11], T(dpix), args[14], deg, args[16], geom, R, binning, img,
                                             False)
        g_or = orc.rasterize_backward(oracle_forward(sc, **kw), dpix)
        floors[tag] = {n: rel_l2(t.cpu().numpy(), g_or[n]) for n, t in zip(GRAD_NAMES, g) if g_or[n].size}
        print(tag, floors[tag])
    with open(path, "w") as f:
        json.dump(floors, f, indent=1)


def main(out_dir):
    ref = build_ref.load_module()
    assert ref is not None, "oracle/_ref/dgr_ref_C.so missing"
    os.makedirs(out_dir, exist_ok=True)
    dev = "cuda:0"
    T = lambda x: torch.as_tensor(np.ascontiguousarray(x), dtype=torch.float32, device=dev)  # noqa: E731
    e = torch.empty(0, device=dev)
    for name, P, dist, W, H, seed, deg in CASES:
        sc = scene_c1(P=P, dist=dist, W=W, H=H, seed=seed)
        a = sc["act"]
        rng = np.random.default_rng(100 + seed)
        sh = a["shs"] if deg == 0 else rng.normal(0, 0.4, (P, (deg + 1) ** 2, 3)).astype(np.float32)
        args = (T(np.ones(3)), T(a["means3D"]), e, T(a["opacities"]), T(a["scales"]), T(a["rotations"]), 1.0, e,
                T(sc["view"]), T(sc["proj"]), float(sc["tanx"]), float(sc["tany"]), H, W, T(sh), deg,
                T(sc["campos"]), False, False)
        R, color, radii, geom, binning, img = ref.rasterize_gaussians(*args)
        dpix = rng.normal(0, 1, (3, H, W)).astype(np.float32)
        g = ref.rasterize_gaussians_backward(args[0], args[1], radii, e, args[4], args[5], 1.0, e, args[8], args[9],
                                             args[10], args[11], T(dpix), args[14], deg, args[16], geom, R, binning,
                                             img, False)
        out = dict(P=P, dist=dist, W=W, H=H, seed=seed, degree=deg, sh=sh if deg else np.zeros(0, np.float32),
                   num_rendered=R, color=color.cpu().numpy(), radii=radii.cpu().numpy(), dL_dcolor=dpix)
        out.update({n: t.cpu().numpy() for n, t in zip(GRAD_NAMES, g)})
        np.savez_compressed(os.path.join(out_dir, f"ref_{name}.npz"), **out)
        print(name, "R =", R, "mean colour", float(color.mean()))
    write_noise_floors(ref, os.path.join(out_dir, os.path.basename(NOISE_FLOORS)))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else "gpurun_out/golden")
