#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Open-DiffusionGS hot path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--dump-outputs DIR]
  (N > 1: launched by the driver as  python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

Metric (BASELINE.json): denoise-steps/s (+ rasterized-views/s) at 256x256.
One "step" = the hot path over one synthetic batch = BASELINE configs[1], the object pipeline:
  1 DiT denoise forward (24 layers, 4 views -> N = 4098 tokens -> P = 262,146 pixel-aligned Gaussians)
  + the 4-view 256x256 splat render of those Gaussians  (DGSDenoiser.forward, denoiser.py:284-287),
random-init weights by the reference's init rules, synthetic image/noise, orbit cameras.

N > 1 (round 2): after the denoise region the SAME launch runs 6 training steps at per-GPU batch 4 and 8 with the overlapped NCCL
gradient all-reduce and again without any, and adds `train: [{samples_per_s, ms_per_step, allreduce_exposed_ms, ...}]` plus
`per_rank` (every rank's step statistics and clocks) to the line.  NCCL's environment is left as the launcher set it.

Prints ONE JSON line (rank 0).  Keys: the driver contract + `roofline` (dominant kernel, live CUDA-event
timing through the library's per-family event hooks) + `cpu_baseline` (oracle on the host cores, bounded
sample) + `e2e` (same metric through the public API with pinned-host inputs, H2D/D2H inside the timed region).
`--dump-outputs DIR` writes what the last timed step returned (the rendered views and the Gaussians) as DIR/<name>.npy in
float32, so that two builds can be compared output for output on the same seeded inputs.
`--impl reference` times the reference's CPU path = the oracle port (the reference has no CPU rasterizer and
its Python package does not import offline; see DESIGN.md) on the host cores.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "open-diffusiongs_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "denoise_steps_per_sec"
UNIT = "steps/s"
H = W = 256
V = 4
PATCH = 8
LAYERS = 24
D = 1024
N_TOK = 2 + V * (H // PATCH) * (W // PATCH)
P_GAUSS = 2 + V * H * W
GAUSSIAN_FIELDS = ("xyz", "features", "scaling", "rotation", "opacity")
DUMP_BYTES = 64 << 20


def dit_forward_flops(n_tok=N_TOK, layers=LAYERS, d=D):
    """SURVEY 8d: F_fwd(N) = L (24 N D^2 + 4 N^2 D + 12 D^2) + 2 (N-2) D (576 + 896)"""
    return layers * (24 * n_tok * d * d + 4 * n_tok * n_tok * d + 12 * d * d) + 2 * (n_tok - 2) * d * (576 + 896)


def attention_flops(n_tok=N_TOK, d=D):
    return 4 * n_tok * n_tok * d  # QK^T + PV, all heads, one layer, one sample


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of each kernel family, from the committed
    `ncu --set full` captures (profiles/r1_ncu_traffic.json); null when a family has no capture."""
    path = os.path.join(ROOT, "profiles", "r1_ncu_traffic.json")
    return json.load(open(path)) if os.path.exists(path) else {}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        j = json.load(open(path))
        return dict(hbm_gbs=j["hbm_gbs"], bf16_tflops=j["bf16_tflops"],
                    bf16_tflops_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------------
# synthetic batch (SURVEY 8d C2), built on the host with fixed seeds
# ------------------------------------------------------------------------------------------------
def make_batch(batch, seed):
    import numpy as np
    import torch
    from dgs_b200 import synth
    rng = np.random.default_rng(seed)
    image = rng.uniform(0, 1, (batch, V, 3, H, W)).astype(np.float32)
    image[:, 1:] = rng.normal(0, 1, (batch, V - 1, 3, H, W)).astype(np.float32)  # views 1..3 are pure noise at t
    c2w, fx = synth.orbit_cameras(V, W, H, radius=3.0, el_deg=20.0)
    c2w = np.broadcast_to(c2w, (batch, V, 4, 4)).copy()
    fx = np.broadcast_to(fx, (batch, V, 4)).copy()
    # rays (TransformInput, systems/utils.py:621-757): pixel centre +0.5, normalised, rotated by c2w
    ys, xs = np.meshgrid(np.arange(H, dtype=np.float32) + 0.5, np.arange(W, dtype=np.float32) + 0.5, indexing="ij")
    ray_o = np.zeros((batch, V, 3, H, W), np.float32)
    ray_d = np.zeros((batch, V, 3, H, W), np.float32)
    for b in range(batch):
        for v in range(V):
            f = fx[b, v]
            d = np.stack([(xs - f[2]) / f[0], (ys - f[3]) / f[1], np.ones_like(xs)], 0)
            d = np.einsum("ij,jhw->ihw", c2w[b, v, :3, :3], d)
            ray_d[b, v] = d / np.linalg.norm(d, axis=0, keepdims=True)
            ray_o[b, v] = c2w[b, v, :3, 3][:, None, None]
    t = np.full((batch,), 500, np.int64)
    tt = torch.from_numpy
    return dict(image=tt(image), ray_o=tt(ray_o), ray_d=tt(ray_d), c2w=tt(c2w), fxfycxcy=tt(fx), t=tt(t))


def dump_outputs(out_dir, arrays, cap=DUMP_BYTES, seed=0):
    """Writes every tensor of `arrays` as out_dir/<name>.npy in float32.  If they come to more than `cap` bytes, every
    array keeps the same fraction of its entries, chosen by a fixed seed (flattened, in index order), so that runs with
    the same arguments write comparable files."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    frac = min(1.0, cap / sum(4 * a.numel() for a in arrays.values()))
    for name, a in arrays.items():
        a = a.detach().float().cpu().numpy()
        if frac < 1.0:
            a = a.ravel()[np.sort(np.random.default_rng(seed).choice(a.size, int(a.size * frac), replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md recipe)
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "250", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (ts, r) in self.rows if t0 <= ts <= t1 + 0.2] or [r for (_, r) in self.rows[-3:]]
        if not rows:
            return None
        sm = [float(r[1]) for r in rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, c in zip(names, r[5:9]) if c.lower().startswith("active")})
        return dict(sm_mhz=statistics.median(sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(rows))


# ------------------------------------------------------------------------------------------------
# CPU baseline: the oracle (reference restatement) on the host cores, bounded sample
# ------------------------------------------------------------------------------------------------
CPU_DIT_LAYERS_SAMPLED = 1
CPU_VIEWS_SAMPLED = 1
_CPU_REF = {}


def cpu_threads():
    """Thread count of every CPU-baseline leg: fixed, so that two records of the same box agree (r1: 0.0159 vs 0.0495
    steps/s with os.cpu_count() threads on a box whose other tenants varied)."""
    return min(os.cpu_count() or 1, 64)


def cpu_reference_step(batch_np=None, threads=None):
    """One BOUNDED sample of the step on the CPU, extrapolated to a full step:
      DiT: fp32 PyTorch oracle at N = 4098 with 1 of the 24 blocks (block time x 24 + measured non-block time),
      rasterizer: C/OpenMP oracle on 1 of the 4 views of the P = 262,146 Gaussians the oracle DiT emits (x 4).
    -> (estimated seconds per full step, detail dict)"""
    import numpy as np
    import torch
    from dgs_b200 import synth
    from oracle import raster as orc
    from oracle.dit import DenoiserOracle
    threads = threads or cpu_threads()
    torch.set_num_threads(threads)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    b = make_batch(1, 0) if batch_np is None else batch_np
    args = (b["image"][:1], b["ray_o"][:1], b["ray_d"][:1], b["t"][:1])
    with torch.no_grad():
        if "m1" not in _CPU_REF:
            torch.manual_seed(0)
            m1 = DenoiserOracle(layers=CPU_DIT_LAYERS_SAMPLED)
            m0 = DenoiserOracle(layers=0)
            m0.load_state_dict({k: v for k, v in m1.state_dict().items() if not k.startswith("transformer.")}, strict=True)
            _CPU_REF.update(m1=m1, m0=m0)
            m1.image_to_gaussians(*(a[..., :64, :64] if a.dim() == 5 else a for a in args))  # lazy-init warm-up
        t0 = time.perf_counter()
        out, _ = _CPU_REF["m1"].image_to_gaussians(*args)
        t_1 = time.perf_counter() - t0
        t0 = time.perf_counter()
        _CPU_REF["m0"].image_to_gaussians(*args)
        t_0 = time.perf_counter() - t0
    t_block = max(t_1 - t_0, 0.0) / CPU_DIT_LAYERS_SAMPLED
    t_dit = t_0 + LAYERS * t_block
    g = {k: v[0].numpy() for k, v in out.items()}
    act = synth.activate(dict(xyz=g["xyz"], features=g["features"], scaling=g["scaling"], rotation=g["rotation"],
                              opacity=g["opacity"]))
    cam = synth.camera_matrices(b["c2w"][0, 0].numpy(), b["fxfycxcy"][0, 0].numpy(), H, W)
    t0 = time.perf_counter()
    st = orc.rasterize_forward(np.ones(3, np.float32), act["means3D"], None, act["opacities"], act["scales"],
                               act["rotations"], 1.0, None, cam[0], cam[1], cam[3], cam[4], H, W, act["shs"], 0, cam[2])
    t_view = time.perf_counter() - t0
    t_step = t_dit + V * t_view
    detail = dict(dit_s=t_dit, dit_block_s=t_block, dit_nonblock_s=t_0, raster_view_s=t_view,
                  instances_per_view=int(st["num_rendered"]), threads=threads, omp_threads=orc.num_threads())
    return t_step, detail


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port) on the host cores."""
    if rank != 0:
        return
    threads = cpu_threads()
    batch = make_batch(1, 0)
    for _ in range(args.warmup):
        cpu_reference_step(batch, threads)
    ts = []
    for _ in range(args.steps):
        t, detail = cpu_reference_step(batch, threads)
        ts.append(t)
    t_step = statistics.mean(ts)
    val = 1.0 / t_step
    sample = (f"per step: fp32 PyTorch oracle DiT at N={N_TOK} with {CPU_DIT_LAYERS_SAMPLED}/{LAYERS} blocks "
              f"(block time x{LAYERS} + non-block time) + C/OpenMP oracle rasterizer on {CPU_VIEWS_SAMPLED}/{V} views "
              f"of P={P_GAUSS} (x{V}); extrapolated to one full step")
    line = dict(impl="reference", metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=t_step * 1e3, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=workload_name(1), per_gpu_batch=1, parallelism="cpu", detail=detail),
                cpu_baseline=dict(value=val, unit=UNIT, cores=threads, kind="port", sample=sample, extrapolated=True),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                views_per_sec=val * V, gpu_launches=0)
    print(json.dumps(line))


class TrainBench:
    """Training step of the obj-256 config (BASELINE configs[2], diffusionGS_rel.yaml: 4 input views, 10 rendered views,
    AdamW lr 1e-5, clip 0.5, EMA 0.9999; loss = the MSE term, fused into the rasterizer -- the LPIPS weights are not available
    offline): one process per GPU, per-GPU batch B, gradients all-reduced over NCCL every step, the per-block buckets
    overlapped with the rest of the backward (dgs_dit_backward_ex block_done events)."""

    def __init__(self, dev, rank, world, render_views, recompute=False, overlap=True, ema=True):
        import torch
        from dgs_b200.denoiser import DGSDenoiser
        from dgs_b200.train import DitTrainer
        self.dev, self.rank, self.world, self.VR, self.overlap = dev, rank, world, render_views, overlap
        torch.manual_seed(0)  # identical initial weights on every rank (what DDP's broadcast establishes)
        self.model = DGSDenoiser(dict(patch_size=PATCH)).to(dev)
        self.trainer = DitTrainer(self.model, lr=1e-5, betas=(0.9, 0.99), eps=1e-8, clip=0.5, recompute=recompute,
                                  overlap_allreduce=overlap, ema_decay=0.9999 if ema else None)
        self.model.train()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        self.host = self.devb = None

    def set_batch(self, B):
        import numpy as np
        import torch
        from dgs_b200 import synth
        VR = self.VR
        host = make_batch(B, seed=self.rank)
        c2w_r, fx_r = synth.orbit_cameras(VR, W, H, radius=3.0, el_deg=20.0, az_step=36.0)
        rng = np.random.default_rng(100 + self.rank)
        host["c2w_r"] = torch.from_numpy(np.broadcast_to(c2w_r, (B, VR, 4, 4)).copy())
        host["fx_r"] = torch.from_numpy(np.broadcast_to(fx_r, (B, VR, 4)).copy())
        host["target"] = torch.from_numpy(rng.uniform(0, 1, (B, VR, 3, H, W)).astype(np.float32))
        self.B = B
        self.host = {k: v.pin_memory() for k, v in host.items()}
        self.devb = {k: v.to(self.dev, non_blocking=True) for k, v in self.host.items()}

    def step(self, b, allreduce=True):
        from dgs_b200 import losses
        out, _ = self.model.image_to_gaussians(b["image"], b["ray_o"], b["ray_d"], b["t"])
        res, _ = losses.fused_render_and_loss(self.model, out, b["c2w_r"], b["fx_r"], H, W, b["target"],
                                              lambdas=dict(lambda_diffusion=1.0))
        self.trainer.overlap = self.overlap and allreduce  # without an all-reduce there is nothing to issue in the backward
        res["loss"].backward()
        self.trainer.optimizer_step(allreduce=allreduce)
        return res["loss"].detach()

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def timed(self, steps, warmup, allreduce=True):
        """-> (max-over-ranks seconds for `steps` steps, this rank's per-step ms, last loss)"""
        import torch
        import torch.distributed as dist
        for _ in range(warmup):
            self.step(self.devb, allreduce)
        self.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b_ in ev:
            self.flush.zero_()
            a.record()
            loss = self.step(self.devb, allreduce)
            b_.record()
        self.barrier()
        step_ms = [a.elapsed_time(b_) for a, b_ in ev]
        total_s = torch.tensor([sum(step_ms) / 1e3], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(total_s, op=dist.ReduceOp.MAX)
        return float(total_s), step_ms, loss


def train_section(dev, rank, world, batches, steps, warmup, render_views):
    """The north-star's data-parallel split measured inside the default bench line (N > 1): per-GPU batch b training
    steps with the overlapped NCCL gradient all-reduce, and the same steps without any all-reduce right after, so that
    the EXPOSED all-reduce time per step is a measured difference.  -> list of dicts (rank 0), one per batch size."""
    import torch
    tb = TrainBench(dev, rank, world, render_views)
    out = []
    for B in batches:
        tb.set_batch(B)
        t_ar, step_ms, loss = tb.timed(steps, warmup, allreduce=True)
        t_no, _, _ = tb.timed(steps, 1, allreduce=False) if world > 1 else (t_ar, None, None)
        out.append(dict(per_gpu_batch=B, global_batch=B * world, samples_per_s=world * B * steps / t_ar,
                        ms_per_step=t_ar / steps * 1e3, ms_per_step_no_allreduce=t_no / steps * 1e3,
                        allreduce_exposed_ms=(t_ar - t_no) / steps * 1e3, steps=steps, warmup=warmup,
                        render_views=render_views, loss=float(loss), step_ms_rank0=[round(v, 2) for v in step_ms],
                        mem_gb=torch.cuda.max_memory_allocated(dev) / 2 ** 30,
                        collective="ncclAllReduce(sum) of 460,391,424 fp32 gradients per step, 3 DiT blocks (227 MB) per call in "
                                   "reverse order on a side stream, gated by the backward's block_done events"))
    del tb
    torch.cuda.empty_cache()
    return out


def run_train(args, rank, local_rank, world):
    """`--workload train`: the training step alone (see TrainBench).  Prints one JSON line (same keys as the default
    workload; `value` = samples/s over all ranks)."""
    import torch
    import torch.distributed as dist
    from dgs_b200 import _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    tb = TrainBench(dev, rank, world, args.render_views, recompute=args.recompute, overlap=not args.no_overlap)
    B, VR = args.batch, args.render_views
    tb.set_batch(B)
    L = _lib.lib()
    sampler = ClockSampler(local_rank)
    for _ in range(args.warmup):
        tb.step(tb.devb)
    if rank == 0:
        sampler.start()
    launches0 = L.dgs_kernel_launch_count()
    t0 = time.time()
    total_s, step_ms, loss = tb.timed(args.steps, 0)
    t1 = time.time()
    launches = L.dgs_kernel_launch_count() - launches0
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    exposed = None
    if world > 1:
        t_no, _, _ = tb.timed(args.steps, 1, allreduce=False)
        exposed = (total_s - t_no) / args.steps * 1e3
    value = world * B * args.steps / total_s
    host, step, barrier = tb.host, tb.step, tb.barrier
    # per-family device time
    L.dgs_profile_enable(1)
    _lib.profile_read()
    for _ in range(args.steps):
        step(tb.devb)
    torch.cuda.synchronize(dev)
    fam = _lib.profile_read()
    L.dgs_profile_enable(0)
    fam_ms = {k: v[0] / args.steps for k, v in fam.items() if v[1]}
    # end to end: pinned host inputs -> device every step, loss read back
    from dgs_b200.diffusion import transform_input
    e2e_keys = [k for k in host if k not in ("ray_o", "ray_d")]  # rays are derived on the device (TransformInput)

    def e2e_step():
        b = {k: host[k].to(dev, non_blocking=True) for k in e2e_keys}
        b["ray_o"], b["ray_d"] = transform_input(b["image"], b["c2w"], b["fxfycxcy"])
        return step(b).to("cpu")
    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tb.flush.zero_()
        lh = e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    line = None
    if rank == 0:
        peaks = load_peaks()
        f_train = 3 * dit_forward_flops() * B  # algorithmic: fwd + 2 x bwd (a recomputed forward is not credited)
        dit_ms = sum(v for k, v in fam_ms.items() if k.startswith("dit."))
        bwd_att = fam_ms.get("dit.bwd_attention")
        roof = None
        if bwd_att:
            ach = 2.5 * attention_flops() * B / (bwd_att / LAYERS * 1e-3) / 1e12  # 5 GEMMs of the algorithm vs 2 forward
            roof = dict(kernel="dit.bwd_attention", bound="tensor", achieved=ach, peak=peaks["bf16_tflops_sustained"],
                        unit="TFLOP/s", frac=ach / peaks["bf16_tflops_sustained"], traffic=None,
                        peak_source=peaks["source"], launch_ms=bwd_att / LAYERS,
                        note="algorithmic FLOPs = 2.5 x forward attention (dV, dP, dQ, dK + S); the kernel pair recomputes S and dP once more")
        line = dict(metric="train-samples/sec @256^2 (DiT fwd+bwd + %d-view render fwd+bwd + grad all-reduce + AdamW+EMA)" % VR,
                    value=value, unit="samples/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                    ms_per_step=total_s / args.steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="bf16", data="synthetic",
                    config=dict(workload="obj-256 train step: 4 input views, %d rendered views, fused MSE loss, AdamW + EMA" % VR,
                                per_gpu_batch=B, activations="recompute" if args.recompute else "stored",
                                parallelism=f"dp{world} (NCCL all-reduce of 460 M fp32 gradients, "
                                            f"{'overlapped per block' if not args.no_overlap else 'after the backward'})",
                                l2="256 MB buffer written between timed steps"),
                    e2e=dict(value=world * B * args.steps / float(e2e_s), unit="samples/s",
                             h2d_bytes_per_step=sum(host[k].numel() * host[k].element_size() for k in e2e_keys),
                             d2h_bytes_per_step=lh.numel() * lh.element_size()),
                    gpu_launches=int(launches), roofline=roof, cpu_baseline=None, clocks=clocks,
                    allreduce_exposed_ms=exposed,
                    breakdown_ms=dict(dit=dit_ms, families={k: round(v, 4) for k, v in fam_ms.items()}),
                    dit_train_tflops=f_train / (dit_ms * 1e-3) / 1e12 if dit_ms else None, loss=float(loss),
                    step_ms=[round(v, 3) for v in step_ms], mem_gb=torch.cuda.max_memory_allocated(dev) / 2 ** 30)
    if world > 1:
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line), flush=True)


def workload_name(batch):
    return (f"obj-256 denoise step (BASELINE configs[1]): 1 DiT forward (24 layers, {N_TOK} tokens) + {V}-view "
            f"256x256 splat render of P={P_GAUSS} Gaussians, per-GPU batch {batch}, random-init weights")


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="samples per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="denoise", choices=["denoise", "train"],
                    help="denoise = BASELINE configs[1] (the contract's default line); train = configs[2]-shaped training "
                         "step (DiT fwd+bwd, V_render-view render fwd+bwd, gradient all-reduce, AdamW)")
    ap.add_argument("--render-views", type=int, default=10)
    ap.add_argument("--recompute", action="store_true", help="train workload: activation recompute (denoiser.py:348-354)")
    ap.add_argument("--no-overlap", action="store_true", help="train workload: all-reduce after the whole backward")
    ap.add_argument("--train-batches", default="4,8", help="per-GPU batch sizes of the training section (N > 1)")
    ap.add_argument("--no-train-section", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (rendered views, Gaussians) as DIR/<name>.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "denoise"):
        ap.error("--dump-outputs applies to the denoise workload of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world == 1:  # the CPU-baseline legs (oracle: torch intra-op + the C oracle's OpenMP team) use a FIXED thread count
        os.environ.setdefault("OMP_NUM_THREADS", str(cpu_threads()))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if args.workload == "train":
        run_train(args, rank, local_rank, world)
        return

    import torch
    import torch.distributed as dist
    from dgs_b200 import _lib
    from dgs_b200.denoiser import DGSDenoiser
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's own environment (NCCL_DEBUG, NCCL_DEBUG_FILE) is left exactly as the launcher set it, so that its log shows
        # the communicator with `world` ranks; the JSON line is the LAST line this process prints.
        dist.init_process_group("nccl", device_id=dev)

    torch.manual_seed(0)
    model = DGSDenoiser(dict(patch_size=PATCH)).to(dev)
    model.packed_weights()
    host = {k: v.pin_memory() for k, v in make_batch(args.batch, seed=rank).items()}
    devb = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    L = _lib.lib()

    keep = bool(args.dump_outputs)
    last_gaussians = {}

    def step(b, keep=False):
        params, _ = model.image_to_gaussians(b["image"], b["ray_o"], b["ray_d"], b["t"])
        if keep:
            last_gaussians.update((k, params[k]) for k in GAUSSIAN_FIELDS)
        return model.render_gaussians(params, b["c2w"], b["fxfycxcy"], H, W)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)  # every rank samples its own GPU (per-rank clocks / power in the N > 1 line);
    sampler.start()                     # started BEFORE the warm-up: spawning nvidia-smi right before the timed region cost the first timed step 5 ms (r2, N = 2)
    for _ in range(args.warmup):
        img = step(devb, keep)  # with --dump-outputs the timed steps keep their Gaussians alive; so do these
    # N > 1: the clocks / power of a box that just went from idle to N busy GPUs settle over the first ~100 ms (r1 SCALE:
    # the first timed region was slower than the later wall-timed e2e loop); extra UNTIMED steps, same on every rank
    for _ in range(30 if world > 1 else 0):
        flush.zero_()
        img = step(devb, keep)
    barrier()

    # ---- timed region 1: inputs resident in HBM, per-step CUDA events, L2 flushed between steps ----

    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = L.dgs_kernel_launch_count()
    barrier()
    t_wall0 = time.time()
    for a, b_ in ev:
        flush.zero_()
        a.record()
        img = step(devb, keep)
        b_.record()
    barrier()
    t_wall1 = time.time()
    # the last timed step's outputs are tensors of their own (not workspace), so the later regions do not overwrite them
    last_outputs = dict(render=img, **last_gaussians) if keep else None
    launches = L.dgs_kernel_launch_count() - launches0
    clocks = sampler.stop(t_wall0, t_wall1)
    step_ms = [a.elapsed_time(b_) for a, b_ in ev]
    total_s = torch.tensor([sum(step_ms) / 1e3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_s, op=dist.ReduceOp.MAX)
    total_s = float(total_s)
    value = world * args.batch * args.steps / total_s
    per_rank = None
    if world > 1:  # where the N-GPU time goes: every rank's own step statistics and clocks during the timed region
        mine = dict(rank=rank, gpu=local_rank, step_ms_min=round(min(step_ms), 3), step_ms_median=round(statistics.median(step_ms), 3),
                    step_ms_max=round(max(step_ms), 3), step_ms_sum=round(sum(step_ms), 3), wall_s=round(t_wall1 - t_wall0, 4),
                    sm_mhz=clocks and clocks["sm_mhz"], reasons=clocks and clocks["reasons"])
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
        per_rank = gathered

    last_R = getattr(model.gs_renderer, "last_num_rendered", None)
    # ---- timed region 2: per-kernel-family device time, same steps with the library's event hooks on ----
    L.dgs_profile_enable(1)
    _lib.profile_read()
    for _ in range(args.steps):
        flush.zero_()
        img = step(devb)
    torch.cuda.synchronize(dev)
    fam = _lib.profile_read()
    L.dgs_profile_enable(0)
    fam_ms = {k: v[0] / args.steps for k, v in fam.items() if v[1]}
    fam_n = {k: v[1] // args.steps for k, v in fam.items() if v[1]}

    # ---- timed region 3: end to end through the public API with pinned HOST buffers ----
    # What the reference pipeline holds on the host is the image and the cameras (pipline_obj.py:267-288); the rays are
    # derived ON THE DEVICE by TransformInput, here dgs_b200.diffusion.transform_input (one kernel).
    from dgs_b200.diffusion import transform_input
    e2e_keys = ("image", "c2w", "fxfycxcy", "t")

    out_host = torch.empty(args.batch, V, 3, H, W, dtype=torch.float32).pin_memory()  # the result lands in pinned memory

    def e2e_step():
        b = {k: host[k].to(dev, non_blocking=True) for k in e2e_keys}
        b["ray_o"], b["ray_d"] = transform_input(b["image"], b["c2w"], b["fxfycxcy"])
        out = step(b)
        out_host.copy_(out, non_blocking=True)
        torch.cuda.current_stream(dev).synchronize()  # the step's result is on the host before the next step starts
        return out_host
    for _ in range(2):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        out_host = e2e_step()
    torch.cuda.synchronize(dev)
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_val = world * args.batch * args.steps / float(e2e_s)
    h2d = sum(host[k].numel() * host[k].element_size() for k in e2e_keys)
    d2h = out_host.numel() * out_host.element_size()

    # ---- N > 1: the training step with the NCCL gradient all-reduce (the path's one collective), same launch ----
    train = None
    if world > 1 and not args.no_train_section:
        del model, devb
        torch.cuda.empty_cache()
        model = None
        train = train_section(dev, rank, world, [int(b) for b in args.train_batches.split(",")], steps=6, warmup=3,
                              render_views=args.render_views)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if last_outputs is not None:
        dump_outputs(args.dump_outputs, last_outputs)

    # ---- roofline of the dominant kernel family ----
    peaks = load_peaks()
    dom = max(fam_ms, key=fam_ms.get) if fam_ms else None
    share = {k: round(v / sum(fam_ms.values()), 4) for k, v in sorted(fam_ms.items(), key=lambda kv: -kv[1])}
    roof = None
    if dom is not None:
        per_launch_ms = fam_ms[dom] / max(fam_n[dom], 1)
        flops = {"dit.attention": attention_flops() * args.batch,
                 "dit.gemm_qkv": 2 * N_TOK * D * 3 * D * args.batch, "dit.gemm_proj": 2 * N_TOK * D * D * args.batch,
                 "dit.gemm_fc1": 2 * N_TOK * D * 4 * D * args.batch, "dit.gemm_fc2": 2 * N_TOK * D * 4 * D * args.batch}
        if dom in flops:
            ach = flops[dom] / (per_launch_ms * 1e-3) / 1e12
            pk = peaks["bf16_tflops_sustained"]
            roof = dict(kernel=dom, bound="tensor", achieved=ach, peak=pk, unit="TFLOP/s", frac=ach / pk,
                        traffic=load_traffic().get(dom),
                        peak_source=peaks["source"] + " (sustained cuBLAS bf16, kernel timed inside a long step)",
                        launch_ms=per_launch_ms, algorithmic_flops_per_launch=flops[dom])
        else:
            # rasterizer family: algorithmic bytes B_fwd = 159 P + 84 R + 20 N_pix per view (SURVEY 8d)
            R = last_R
            nbytes = None if R is None else (159 * P_GAUSS * V + 84 * R + 20 * H * W * V) * args.batch
            tot_ms = sum(v for k, v in fam_ms.items() if k.startswith("raster."))
            ach = None if nbytes is None else nbytes / (tot_ms * 1e-3) / 1e9
            roof = dict(kernel=dom, bound="hbm", achieved=ach, peak=peaks["hbm_gbs"], unit="GB/s",
                        frac=None if ach is None else ach / peaks["hbm_gbs"], traffic=None,
                        peak_source=peaks["source"], launch_ms=per_launch_ms, note="whole rasterizer forward vs B_fwd")
    dit_ms = sum(v for k, v in fam_ms.items() if k.startswith("dit."))
    ras_ms = sum(v for k, v in fam_ms.items() if k.startswith("raster."))

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = cpu_threads()
        t_cpu, detail = min((cpu_reference_step(None, threads) for _ in range(2)), key=lambda r: r[0])
        cpu = dict(value=1.0 / t_cpu, unit=UNIT, cores=threads, kind="port", extrapolated=True,
                   sample=(f"best of 2 bounded samples, EXTRAPOLATED to a full step: fp32 PyTorch oracle DiT with "
                           f"{CPU_DIT_LAYERS_SAMPLED}/{LAYERS} blocks timed (x{LAYERS} + non-block time) + C/OpenMP oracle "
                           f"rasterizer on 1/{V} views (x{V}); dit {detail['dit_s']:.1f}s + raster {V}x{detail['raster_view_s']:.1f}s; "
                           f"{threads} threads (pinned: min(os.cpu_count(), 64))"),
                   detail=detail)

    ms_per_step = total_s / args.steps * 1e3
    line = dict(
        metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=args.warmup,
        ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
        data="synthetic",
        config=dict(workload=workload_name(args.batch), per_gpu_batch=args.batch, parallelism=f"replicas x{world}",
                    l2="256 MB buffer written between timed steps (L2 flush); bf16 weights alone are 0.92 GB > 126 MB L2",
                    dit_dtype="bf16 tensor-core GEMM/attention, fp32 residual/LN/softmax", raster_dtype="f32"),
        views_per_sec=value * V,
        e2e=dict(value=e2e_val, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h),
        gpu_launches=int(launches),
        roofline=roof, cpu_baseline=cpu, clocks=clocks,
        breakdown_ms=dict(dit=dit_ms, raster=ras_ms, families={k: round(v, 4) for k, v in fam_ms.items()},
                          share=share, launches_per_step=fam_n),
        dit_tflops=dit_forward_flops() * args.batch / (dit_ms * 1e-3) / 1e12 if dit_ms else None,
        step_ms_min=min(step_ms), step_ms_max=max(step_ms), step_ms=[round(v, 3) for v in step_ms],
    )
    if per_rank is not None:
        line["per_rank"] = per_rank
    if train is not None:
        line["train"] = train
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
