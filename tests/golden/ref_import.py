"""Loads the REFERENCE's own Python modules by path from /root/reference, with stub modules standing in for the
third-party packages this image lacks, so that tests and the golden-vector scripts can execute the reference's code
itself (not a restatement).  Test infrastructure; nothing in the product path imports it, and it only works where
/root/reference is mounted (this container -- not the GPU box, which uses the fixtures committed next to this file).

What is real and what is a stub:

  real (executed from /root/reference, unmodified)
    diffusionGS/models/denoiser/denoiser.py            DGSDenoiser, TimestepEmbedder, GaussiansUpsampler, ImageTokenDecoder
    diffusionGS/models/denoiser/denoiser_scene.py      DGSDenoiser (scene twin)
    diffusionGS/models/transformers/utils_transformer.py   DiTBlock, modulate, _init_weights
    diffusionGS/models/gsrenderer/gs_core.py           Camera, GaussianModel, render_opencv_cam, DeferredGaussianRender
    diffusionGS/models/gsrenderer/renderer.py          Renderer
    submodules/diff-gaussian-rasterization/diff_gaussian_rasterization/__init__.py   the binding classes

  stubs (absent offline; see SURVEY section 0.3)
    timm.models.vision_transformer   Attention / Mlp / PatchEmbed: timm==0.9.16 (requirement.txt:25) is not vendored.
        Its published forward is restated HERE independently of oracle/dit.py (fused path:
        F.scaled_dot_product_attention, as timm 0.9.16 does when `use_fused_attn()`), so the oracle's explicit
        softmax(q k^T / sqrt(d)) v is cross-checked against torch's SDPA.
    xformers.ops, easydict, plyfile, imageio, kiui, trimesh, matplotlib      import-only stubs (never called on the path)
    diffusionGS (package), diffusionGS.utils.{base,typing,checkpoint,ops,mesh_utils}   registry + BaseModule skeleton
        (BaseModule.__init__ = dataclass Config from a dict + configure(), utils/base.py:88-117)
    diff_gaussian_rasterization._C   the compiled extension: backed by the CPU oracle (oracle/raster.py, itself pinned
        against the reference's CUDA kernels by tests/golden/ref_*.npz) with the extension's exact argument tuples
        (rasterize_points.cu:35-196), so the reference's binding, gs_core.py and renderer.py run on CPU tensors.
"""
import dataclasses
import importlib.util
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

REF = os.environ.get("DGS_REFERENCE_ROOT", "/root/reference")
DGR = os.path.join(REF, "submodules", "diff-gaussian-rasterization")


def available() -> bool:
    return os.path.isfile(os.path.join(REF, "diffusionGS", "models", "denoiser", "denoiser.py"))


# ----------------------------------------------------------------------------------------------- timm 0.9.16 stub
class _TimmAttention(nn.Module):
    """timm 0.9.16 vision_transformer.Attention (qk_norm=False, drops 0), fused-attention branch."""

    def __init__(self, dim, num_heads=8, qkv_bias=False, qk_norm=False, attn_drop=0.0, proj_drop=0.0, norm_layer=nn.LayerNorm):
        super().__init__()
        assert dim % num_heads == 0 and not qk_norm
        self.num_heads = num_heads
        self.head_dim = dim // num_heads
        self.scale = self.head_dim ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.q_norm, self.k_norm = nn.Identity(), nn.Identity()
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)

    def forward(self, x):
        B, N, C = x.shape
        qkv = self.qkv(x).reshape(B, N, 3, self.num_heads, self.head_dim).permute(2, 0, 3, 1, 4)
        q, k, v = qkv.unbind(0)
        q, k = self.q_norm(q), self.k_norm(k)
        x = F.scaled_dot_product_attention(q, k, v, dropout_p=0.0)
        x = x.transpose(1, 2).reshape(B, N, C)
        return self.proj_drop(self.proj(x))


class _TimmMlp(nn.Module):
    """timm 0.9.16 layers.Mlp (bias=True, norm_layer=None, use_conv=False)."""

    def __init__(self, in_features, hidden_features=None, out_features=None, act_layer=nn.GELU, norm_layer=None, bias=True,
                 drop=0.0, use_conv=False):
        super().__init__()
        out_features = out_features or in_features
        hidden_features = hidden_features or in_features
        self.fc1 = nn.Linear(in_features, hidden_features, bias=bias)
        self.act = act_layer()
        self.drop1 = nn.Dropout(drop)
        self.norm = nn.Identity()
        self.fc2 = nn.Linear(hidden_features, out_features, bias=bias)
        self.drop2 = nn.Dropout(drop)

    def forward(self, x):
        return self.drop2(self.fc2(self.norm(self.drop1(self.act(self.fc1(x))))))


class _EasyDict(dict):
    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    __getattr__ = dict.__getitem__
    __setattr__ = dict.__setitem__


# ----------------------------------------------------------------------------------------------- _C on the CPU oracle
class _OracleC:
    """`diff_gaussian_rasterization._C` with the extension's signatures (ext.cpp:15-19), arithmetic = oracle/raster.py."""

    def __init__(self):
        self._states = {}

    @staticmethod
    def _np(t):
        return t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else t

    def rasterize_gaussians(self, bg, means3D, colors, opacity, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix,
                            projmatrix, tanfovx, tanfovy, image_height, image_width, sh, degree, campos, prefiltered, debug):
        from oracle import raster as R
        if means3D.dim() != 2 or means3D.shape[1] != 3:
            raise RuntimeError("means3D must have dimensions (num_points, 3)")
        n = self._np
        st = R.rasterize_forward(n(bg), n(means3D), n(colors), n(opacity), n(scales), n(rotations), float(scale_modifier),
                                 n(cov3D_precomp), n(viewmatrix), n(projmatrix), float(tanfovx), float(tanfovy),
                                 int(image_height), int(image_width), n(sh), int(degree), n(campos))
        h = len(self._states)
        self._states[h] = st
        handle = torch.tensor([h], dtype=torch.int64)
        e = torch.empty(0, dtype=torch.uint8)
        return (int(st["num_rendered"]), torch.from_numpy(st["color"].copy()), torch.from_numpy(st["radii"].copy()), handle, e, e)

    def rasterize_gaussians_backward(self, bg, means3D, radii, colors, scales, rotations, scale_modifier, cov3D_precomp, viewmatrix,
                                     projmatrix, tanfovx, tanfovy, dL_dout_color, sh, degree, campos, geomBuffer, R_, binningBuffer,
                                     imgBuffer, debug):
        from oracle import raster as R
        g = R.rasterize_backward(self._states[int(geomBuffer[0])], self._np(dL_dout_color.contiguous()))
        t = lambda k: torch.from_numpy(g[k])  # noqa: E731
        return (t("dL_dmeans2D"), t("dL_dcolors"), t("dL_dopacity"), t("dL_dmeans3D"), t("dL_dcov3D"), t("dL_dsh"),
                t("dL_dscales"), t("dL_drotations"))

    def mark_visible(self, means3D, viewmatrix, projmatrix):
        from oracle import raster as R
        return torch.from_numpy(R.mark_visible(self._np(means3D), self._np(viewmatrix)))


# ----------------------------------------------------------------------------------------------- module plumbing
def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    if "." not in name or name.count(".") < 9:
        m.__path__ = []  # behaves as a package: `import a.b.c` resolves through sys.modules
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], child, m)
    return m


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    sys.modules[name] = m
    parent, _, child = name.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], child, m)
    spec.loader.exec_module(m)
    return m


class _BaseModule(nn.Module):
    """Skeleton of diffusionGS/utils/base.py:88-117: cfg = structured Config built from a dict, then configure()."""

    @dataclasses.dataclass
    class Config:
        weights: object = None

    def __init__(self, cfg=None, *args, **kwargs):
        super().__init__()
        fields = {f.name for f in dataclasses.fields(self.Config)}
        cfg = dict(cfg or {})
        unknown = set(cfg) - fields
        if unknown:
            raise KeyError(f"unknown config keys {sorted(unknown)}")  # omegaconf structured configs reject them too
        self.cfg = self.Config(**cfg)
        self.configure(*args, **kwargs)
        self.register_buffer("_dummy", torch.zeros(0).float(), persistent=False)

    def configure(self, *args, **kwargs):
        pass


_loaded = {}


def load(renderer="stub"):
    """-> namespace with the reference modules.  renderer = "stub" (a no-op nn.Module: DiT-only checks) or "oracle"
    (the reference's gs_core.py / renderer.py / binding running on the CPU oracle's `_C`)."""
    if renderer in _loaded:
        return _loaded[renderer]
    if not available():
        raise RuntimeError(f"{REF} is not mounted")
    root = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    if root not in sys.path:
        sys.path.insert(0, root)
    for k in [k for k in sys.modules if k == "diffusionGS" or k.startswith("diffusionGS.") or
              k.startswith("diff_gaussian_rasterization")]:
        del sys.modules[k]
    registry = {}

    def register(name):
        def deco(cls):
            registry[name] = cls
            return cls
        return deco

    _mod("easydict", EasyDict=_EasyDict)
    _mod("xformers")
    _mod("xformers.ops")
    _mod("timm")
    _mod("timm.models")
    _mod("timm.models.vision_transformer", Attention=_TimmAttention, Mlp=_TimmMlp, PatchEmbed=nn.Identity)
    _mod("diffusionGS", register=register, find=registry.__getitem__, __modules__=registry)
    for pkg in ("models", "models.transformers", "models.gsrenderer", "models.denoiser", "utils"):
        _mod("diffusionGS." + pkg)
    import typing
    ty = {k: getattr(typing, k) for k in typing.__all__}
    ty.update(Tensor=torch.Tensor, Float=typing.Any, Int=typing.Any, Bool=typing.Any, Num=typing.Any, DictConfig=dict)
    _mod("diffusionGS.utils.typing", __all__=list(ty), **ty)
    _mod("diffusionGS.utils.base", BaseModule=_BaseModule)
    _mod("diffusionGS.utils.checkpoint", checkpoint=torch.utils.checkpoint.checkpoint)
    _mod("diffusionGS.utils.ops", generate_dense_grid_points=None)
    _mod("diffusionGS.utils.mesh_utils", decimate_mesh=None, clean_mesh=None)
    ns = types.SimpleNamespace(registry=registry)
    ns.utils_transformer = _load("diffusionGS.models.transformers.utils_transformer",
                                 os.path.join(REF, "diffusionGS/models/transformers/utils_transformer.py"))
    if renderer == "stub":
        class Renderer(nn.Module):
            def __init__(self, config):
                super().__init__()
                self.config = config
        _mod("diffusionGS.models.gsrenderer.renderer", Renderer=Renderer, SceneRenderer=Renderer)
    else:
        for name in ("matplotlib", "plyfile", "imageio", "kiui", "trimesh"):
            if name not in sys.modules:
                try:
                    importlib.import_module(name)
                except ImportError:
                    _mod(name, PlyData=None, PlyElement=None)
        pkg = _mod("diff_gaussian_rasterization")
        pkg.__path__ = [os.path.join(DGR, "diff_gaussian_rasterization")]
        ns.C = _OracleC()
        sys.modules["diff_gaussian_rasterization._C"] = ns.C
        pkg._C = ns.C
        src = os.path.join(DGR, "diff_gaussian_rasterization", "__init__.py")
        spec = importlib.util.spec_from_file_location("diff_gaussian_rasterization", src,
                                                      submodule_search_locations=pkg.__path__)
        binding = importlib.util.module_from_spec(spec)
        binding._C = ns.C
        sys.modules["diff_gaussian_rasterization"] = binding
        sys.modules["diff_gaussian_rasterization._C"] = ns.C
        spec.loader.exec_module(binding)
        ns.binding = binding
        ns.gs_core = _load("diffusionGS.models.gsrenderer.gs_core", os.path.join(REF, "diffusionGS/models/gsrenderer/gs_core.py"))
        ns.renderer = _load("diffusionGS.models.gsrenderer.renderer", os.path.join(REF, "diffusionGS/models/gsrenderer/renderer.py"))
    ns.denoiser = _load("diffusionGS.models.denoiser.denoiser", os.path.join(REF, "diffusionGS/models/denoiser/denoiser.py"))
    ns.denoiser_scene = _load("diffusionGS.models.denoiser.denoiser_scene",
                              os.path.join(REF, "diffusionGS/models/denoiser/denoiser_scene.py"))
    _loaded[renderer] = ns
    return ns


class cpu_device_shim:
    """gs_core.py:889-891 allocates `screenspace_points` with device="cuda".  On a box without a GPU the golden script
    runs the reference's renderer on CPU tensors; this context manager maps that one literal to the CPU."""

    def __enter__(self):
        self._orig = torch.empty_like

        def empty_like(t, *a, **kw):
            if kw.get("device") == "cuda" and not torch.cuda.is_available():
                kw["device"] = t.device
            return self._orig(t, *a, **kw)
        torch.empty_like = empty_like
        return self

    def __exit__(self, *exc):
        torch.empty_like = self._orig


def seeded(shape, seed, scale=1.0):
    return torch.from_numpy(np.random.default_rng(seed).normal(0, scale, shape).astype(np.float32))


def seeded_state_dict(module, seed):
    """Deterministic, non-degenerate parameters for `module` (same values on every box: numpy Generator streams are
    stable): matrices ~ N(0, 1/fan_in) so activations stay O(1) through the depth, biases / adaLN biases ~ N(0, 0.1^2)
    (the reference's zero-initialised biases would leave those code paths untested), LayerNorm weights 1 + N(0, 0.1^2),
    the Gaussian position embedding ~ N(0, 1)."""
    return seeded_params({k: tuple(v.shape) for k, v in module.state_dict().items()}, seed)


def seeded_params(shapes, seed):
    """seeded_state_dict for an ordered {name: shape}; the values depend on the order of the names."""
    rng = np.random.default_rng(seed)
    sd = {}
    for k, shape in shapes.items():
        if k.endswith("layernorm.weight"):
            a = 1.0 + 0.1 * rng.standard_normal(shape)
        elif k.endswith(".bias"):
            a = 0.1 * rng.standard_normal(shape)
        elif k == "gaussians_pos_embedding":
            a = rng.standard_normal(shape)
        else:
            a = rng.standard_normal(shape) / np.sqrt(shape[-1])
        sd[k] = torch.from_numpy(a.astype(np.float32))
    return sd


def seeded_dit_inputs(b, v, h, w, seed):
    """images in [0,1], ray origins on a shell of radius ~2, unit ray directions, integer timesteps."""
    rng = np.random.default_rng(seed)
    img = torch.from_numpy(rng.random((b, v, 3, h, w)).astype(np.float32))
    ro = torch.from_numpy((rng.standard_normal((b, v, 3, 1, 1)) * 1.2).astype(np.float32)).expand(b, v, 3, h, w).contiguous()
    rd = torch.from_numpy(rng.standard_normal((b, v, 3, h, w)).astype(np.float32))
    rd = rd / rd.norm(dim=2, keepdim=True)
    t = torch.from_numpy(rng.integers(0, 1000, size=(b,)).astype(np.int64))
    return img, ro, rd, t


# name -> (scene, ray_pe_type, model config, (b, v, h, w), seed).  "s*" = small width (CPU oracle pin, seconds);
# "w1024_*" = the product's width with 2 blocks (GPU parity against numbers produced by the reference's own code).
DIT_CASES = {
    "s_obj_rel": (False, "relative_plk", dict(width=64, dim_heads=16, num_layers=2, patch_size=8), (2, 2, 16, 16), 11),
    "s_obj_plk": (False, "plk", dict(width=64, dim_heads=16, num_layers=2, patch_size=8), (2, 2, 16, 16), 12),
    "s_scene_plk": (True, "plk", dict(width=64, dim_heads=16, num_layers=3, patch_size=8), (1, 3, 16, 24), 13),
    "s_scene_rel": (True, "relative_plk", dict(width=64, dim_heads=16, num_layers=2, patch_size=4), (2, 1, 8, 8), 14),
    "w1024_obj_rel": (False, "relative_plk", dict(width=1024, dim_heads=64, num_layers=2, patch_size=8), (2, 2, 32, 32), 21),
    "w1024_scene_plk": (True, "plk", dict(width=1024, dim_heads=64, num_layers=2, patch_size=8), (1, 3, 32, 48), 22),
    "w1024_obj_plk": (False, "plk", dict(width=1024, dim_heads=64, num_layers=2, patch_size=8), (1, 2, 32, 32), 23),
}
GS_KEYS = ("xyz", "features", "scaling", "rotation", "opacity")
SKETCH_BUCKETS = 32


def sketch(x, seed=7):
    """Count sketch of a tensor: every entry is added, with a fixed random sign, to one of SKETCH_BUCKETS fixed random
    buckets.  For a stored reference r and a candidate x, |sketch(x) - sketch(r)| estimates |x - r| (relative spread
    ~ 1/sqrt(2 * SKETCH_BUCKETS)) from every entry, where storing r itself would take megabytes."""
    x = np.asarray(x.detach() if isinstance(x, torch.Tensor) else x, np.float64).ravel()
    rng = np.random.default_rng(seed)
    bucket = rng.integers(0, SKETCH_BUCKETS, x.size)
    sign = rng.integers(0, 2, x.size) * 2.0 - 1.0
    return np.bincount(bucket, weights=sign * x, minlength=SKETCH_BUCKETS)


def sketched_rel(x, ref_sketch, ref_norm, seed=7):
    """Estimate of |x - r| / |r| from r's sketch and norm."""
    return float(np.linalg.norm(sketch(x, seed) - ref_sketch) / (ref_norm + 1e-30))


def reference_dit_case(name):
    """Runs the reference's own DGSDenoiser (object or scene twin) on the case's seeded parameters and inputs.
    -> (model, inputs, outputs dict incl. img_aligned_xyz, parameter-gradient dict of the seeded scalar loss)."""
    scene, pe, cfg, (b, v, h, w), seed = DIT_CASES[name]
    ns = load("stub")
    cls = (ns.denoiser_scene if scene else ns.denoiser).DGSDenoiser
    model = cls(dict(cfg, in_channels=9, n_gaussians=2, ray_pe_type=pe))
    model.load_state_dict(seeded_state_dict(model, seed), strict=True)
    img, ro, rd, t = seeded_dit_inputs(b, v, h, w, seed + 1000)
    out, ia = model.image_to_gaussians(img, ro, rd, t)
    outs = {k: out[k] for k in GS_KEYS}
    outs["img_aligned_xyz"] = ia
    cot = {k: seeded(tuple(o.shape), seed + 2000 + i) for i, (k, o) in enumerate(outs.items()) if k != "img_aligned_xyz"}
    loss = sum((outs[k] * cot[k]).sum() for k in cot)
    grads = torch.autograd.grad(loss, list(model.parameters()))
    grads = {k: g for (k, _), g in zip(model.named_parameters(), grads)}
    return model, (img, ro, rd, t), {k: o.detach() for k, o in outs.items()}, grads, cot
