"""Writes tests/golden/dit_ref_<case>.npz: outputs of the REFERENCE's own denoiser code (denoiser.py /
denoiser_scene.py / utils_transformer.py executed from /root/reference through tests/golden/ref_import.py) on seeded
parameters and inputs.  Parameters and inputs are regenerated from the seed on any box (ref_import.seeded_*), so the
fixtures hold only the outputs and a digest of the gradients.

Also writes tests/golden/dit_ref_pins.npz, what tests/test_oracle_dit_vs_reference.py holds the oracle to beyond those
outputs: per pinned case the reference's parameter names and shapes in state_dict order (the order fixes the seeded
values) with the norm and the count sketch of every parameter gradient, and per building block the same names with the
block's output.

    DGS_REFERENCE_ROOT=<checkout of the reference> python tests/golden/make_dit_golden.py
"""
import hashlib
import os
import sys
from types import SimpleNamespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_import as ri  # noqa: E402

PINNED = [n for n in ri.DIT_CASES if n.startswith("s_")] + ["w1024_obj_rel"]
PINS = os.path.join(HERE, "dit_ref_pins.npz")
BLOCK_WIDTH, BLOCK_HEADS = 128, 4


def block_inputs():
    """tokens x [2, 37, width], conditioning c [2, width], timesteps t [2]"""
    return ri.seeded((2, 37, BLOCK_WIDTH), 3), ri.seeded((2, BLOCK_WIDTH), 4), torch.tensor([3, 977])


def reference_blocks():
    """-> {name: (reference module, its arguments)}"""
    ns = ri.load("stub")
    D, H = BLOCK_WIDTH, BLOCK_HEADS
    x, c, t = block_inputs()
    return {"DiTBlock": (ns.utils_transformer.DiTBlock(D, H), (x, c)),
            "TimestepEmbedder": (ns.denoiser.TimestepEmbedder(D), (t,)),
            "GaussiansUpsampler": (ns.denoiser.GaussiansUpsampler(SimpleNamespace(width=D, gaussians_sh_degree=0)), (x, c)),
            "ImageTokenDecoder": (ns.denoiser.ImageTokenDecoder(SimpleNamespace(width=D, gaussians_sh_degree=0, patch_size=4)),
                                  (x, c))}


def _pack_shapes(sd):
    return np.array([k + ":" + ",".join(str(n) for n in v.shape) for k, v in sd.items()])


def shapes(z, prefix):
    """The ordered {parameter name: shape} stored as `prefix`/shapes in a pins file."""
    return {k: tuple(int(n) for n in s.split(",") if n) for k, s in (e.split(":") for e in z[prefix + "/shapes"])}


def gradient_digests(z, case):
    """-> {parameter name: (count sketch, norm)} of the reference's gradients in a pins file."""
    return {k: (s, float(n)) for k, s, n in zip(z[case + "/grad_names"], z[case + "/gsketch"], z[case + "/gnorm"])}


def main():
    torch.set_num_threads(8)
    for name in ri.DIT_CASES:
        model, _, outs, grads, _ = ri.reference_dit_case(name)
        rec = {"out/" + k: v.numpy() for k, v in outs.items()}
        # gradient digest: per-parameter L2 norm and a fixed random projection (a full copy would be 100 MB at width 1024)
        rng = np.random.default_rng(7)
        for k, g in grads.items():
            gg = g.double().numpy().ravel()
            rec["gnorm/" + k] = np.float64(np.linalg.norm(gg))
            rec["gproj/" + k] = np.float64(gg @ rng.standard_normal(gg.size))
        path = os.path.join(HERE, f"dit_ref_{name}.npz")
        np.savez_compressed(path, **rec)
        print(name, {k: tuple(v.shape) for k, v in outs.items()}, os.path.getsize(path), "bytes")
    write_pins()


def write_pins():
    torch.set_num_threads(8)
    rec = {}
    for name in PINNED:
        model, _, outs, grads, _ = ri.reference_dit_case(name)
        rec[f"{name}/shapes"] = _pack_shapes(model.state_dict())
        rec[f"{name}/grad_names"] = np.array(list(grads))
        rec[f"{name}/gnorm"] = np.array([np.linalg.norm(g.double().numpy()) for g in grads.values()])
        rec[f"{name}/gsketch"] = np.stack([ri.sketch(g) for g in grads.values()])
    with torch.no_grad():
        for name, (ref, args) in reference_blocks().items():
            sd = ri.seeded_state_dict(ref, 5)
            ref.load_state_dict(sd, strict=True)
            rec[f"blocks/{name}/shapes"] = _pack_shapes(sd)
            rec[f"blocks/{name}/out"] = ref(*args).numpy()
        x, c, _ = block_inputs()
        rec["blocks/modulate_sha256"] = np.array(hashlib.sha256(ri.load("stub").utils_transformer.modulate(x, c, 2 * c)
                                                                .numpy().tobytes()).hexdigest())
    np.savez_compressed(PINS, **rec)
    print(PINS, os.path.getsize(PINS), "bytes")


if __name__ == "__main__":
    main()
