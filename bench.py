#!/usr/bin/env python
"""bench.py - training rays/s of the LiDAR4D hot path on B200 (driver contract in the task brief).

Workload (BASELINE.json configs[1]): synthetic KITTI-360-like sweep of 64x1024 rays x 768 samples,
L=16 4D hash + 6 hex-planes + flow field, 50-frame straight trajectory (SURVEY.md 8(d)).
One "step" = one optimiser step on one 65,536-ray sweep of one frame: forward + backward of the
fused kernels over the sweep (in ray chunks, gradients accumulated), one Adam step with the
reference's recipe (main_lidar4d.py:298-300) and the re-staging of the kernel working set.

  python bench.py [--gpus N --steps K --warmup W]            this repo's CUDA path
  python bench.py --impl reference [...]                     CPU reference arm: the oracle port of the
                                                             reference python path (tiny-cuda-nn cannot run
                                                             anywhere here), bounded sample per step
Under torchrun (N>1) every rank renders its own sweep (weak scaling, rays shard with no data-path
collective) and the flat gradient arena is all-reduced once per step over NCCL.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H_SWEEP, W_SWEEP, S_STEPS, N_FRAMES = 64, 1024, 768, 50


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--levels", type=int, default=16, help="n_levels_hash (BASELINE configs[1]: L=16; reference default 8)")
    ap.add_argument("--ray-batch", type=int, default=16384, help="rays per fused forward/backward launch")
    ap.add_argument("--rays", type=int, default=H_SWEEP * W_SWEEP, help="rays per step (sweep size)")
    ap.add_argument("--cpu-rays", type=int, default=64, help="rays of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every rank renders --rays rays per step; strong: --rays is the GLOBAL batch, sharded over the ranks "
                         "(BASELINE.json configs[2]: --scaling strong --rays 4096)")
    ap.add_argument("--mode", default="train", choices=["train", "infer"],
                    help="infer: BASELINE.json configs[3], forward-only render of one 64x2048 frame per step")
    ap.add_argument("--eager-rays", type=int, default=1024,
                    help="rays per step of the GPU-eager baseline leg (the reference's op graph in plain torch under fp16 autocast); 0 = skip")
    ap.add_argument("--streams", type=int, default=1,
                    help="CUDA streams the ray chunks of a step alternate over: the latency-bound tensor-core kernels of one chunk "
                         "overlap the L1TEX/LSU-bound gather / scatter kernels of the next (1 = serial)")
    ap.add_argument("--loss", default="unit", choices=["unit", "main"],
                    help="unit: |depth-0.3| + (image-0.5)^2 with unit weights (the synthetic loss of round 1); main: the reference's main "
                         "loss with its weights (alpha_d 1, alpha_r 0.01, alpha_i 0.1, label smoothing) through lidar4d_b200.losses")
    ap.add_argument("--pipeline", default="split", choices=["split", "fused"])
    ap.add_argument("--mlp", default="fp16", choices=["fp16", "fp32"],
                    help="fp16: MLP weights as fp16 working copies (as tiny-cuda-nn), tensor-core dense kernels; fp32: FMA")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed to DIR/<name>.npy (rank 0): the depth "
                         "and image of every ray, the loss and, when training, a fixed sample of the gradients and updated "
                         "parameters; the inputs depend on the arguments only, so two builds can be compared file for file")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


def model_kwargs(levels):
    return dict(n_levels_hash=levels, num_frames=N_FRAMES + 1, near_lidar=0.0105, far_lidar=0.851)


def randomize(model, seed=0):
    """SURVEY.md 8(d) parameters: hash tables U(-0.5,0.5), planes reference init + N(0,0.1), flow head N(0,1e-3)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    with torch.no_grad():
        for k, p in model.named_parameters():
            if "hash" in k or "grid_enc" in k:
                n = p.numel()
                chunk = torch.rand(min(n, 1 << 22), generator=g) - 0.5
                reps = (n + chunk.numel() - 1) // chunk.numel()
                p.copy_(chunk.repeat(reps)[:n].view_as(p).to(p.device))
            elif "planes" in k:
                p.add_((torch.randn(p.shape, generator=g) * 0.1).to(p.device))


def kernel_bytes(cfg):
    """Algorithmic bytes per sample of every kernel of the pipeline (DESIGN.md 4.3)."""
    L, D = cfg.n_levels_hash, cfg.sigma_in_dim
    planes = 4 * 3 * 4 * 32
    # gather: static hash 8 B x 8 corners; dynamic hash from the per-launch contracted tables: 4 B x 4 corners x 3 planes x 3 queries
    # (round 1: 16-byte pair records); flow grid; static planes 4 texels, time planes 2 texels of a contracted row x 3 queries
    gather = L * 8 * 8 + 3 * 3 * L * 4 * 4 + 8 * 8 * 16 + 4 * 3 * (4 * 32) + 4 * 3 * 3 * (2 * 32)
    fwd, bwd = algorithmic_bytes(cfg)
    exch = 4 * (D + 16 + 6)
    return {
        "forward": fwd, "backward": bwd, "k_render_fwd": fwd, "k_render_bwd": bwd,
        "k_fwd_gather": gather + exch,                                     # table/plane gathers + feature / flow planes written
        "k_fwd_flow": 8 * 8 * 16 + 4 * 22,                                 # flow-grid gather + flow-in / flow planes written
        "k_fwd_dense": 4 * D + 12,                                          # features read, sigma/attr saved
        "k_bwd_dense": 2 * 4 * D + 4 * D + 12,                              # features read twice, dfeat written
        # dynamic hash: one fp32 per entry read-modify-written (scalar accumulators); plane gradients (static 4 texels, time rows
        # 2 texels x 3 queries) read-modify-written + the same texels read for the product rule; dfeat read, dflow written
        "k_bwd_scatter": 2 * (3 * L * 4 * 4 + 4 * 3 * 4 * 32 + 4 * 3 * 3 * 2 * 32) + (4 * 3 * 4 * 32 + 4 * 3 * 3 * 2 * 32) + 4 * (D - 4 * L) + 48,
        "k_bwd_scatter_static": 2 * (L * 8 * 16) + 4 * 4 * L,
        "k_bwd_flow": 4 * 22 + 4 * 16,                                       # dflow + flow-in read, dfin written
        "k_bwd_flowgrid": 2 * (8 * 8 * 32) + 4 * 16,
    }


def algorithmic_bytes(cfg):
    """Per-sample algorithmic bytes (SURVEY.md 8(d), restated for this configuration in DESIGN.md)."""
    L = cfg.n_levels_hash
    fwd = L * 8 * 8 + 3 * (3 * 2 * L * 4 * 8) + 8 * 8 * 16 + 4 * 3 * 4 * 32 + 3 * (4 * 3 * 4 * 32)
    scatter = L * 8 * 16 + 3 * 2 * L * 4 * 16 + 8 * 8 * 32 + (4 * 3 * 4 * 32) * 4
    bwd = 2 * scatter + 4 * (4 * 3 * 4 * 32) + 4 * (cfg.sigma_in_dim + 16 + 3)
    return fwd, bwd


class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.strip().split(",") for r in open(self.path) if r.strip()]
            sm = [float(r[0]) for r in rows]
            out["samples"] = len(sm)
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(rows[0][1])
                out["power_w_max"] = max(float(r[2]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for i, n in enumerate(names):
                    if any("Active" in r[3 + i] and "Not" not in r[3 + i] for r in rows):
                        out["reasons"].append(n)
            os.unlink(self.path)
        except Exception:
            pass
        return out


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# =============================================================================
# CPU arm: the oracle port of the reference python path
# =============================================================================
def reference_main_loss(out):
    """The bench's synthetic loss as a torch op chain - what the baseline legs time (same work as either --loss choice of
    the CUDA arm: an L1 on depth and an MSE on the two image channels)."""
    return (out["depth_lidar"] - 0.3).abs().mean() + ((out["image_lidar"] - 0.5) ** 2).mean()


def cpu_reference_step(orc, opt, ro, rd, t, seed):
    from oracle import lidar4d_oracle as O  # noqa: F401  (bench cpu_baseline / --impl reference leg only)
    opt.zero_grad()
    out = orc.render(torch.from_numpy(ro), torch.from_numpy(rd), t, num_steps=S_STEPS, perturb=True, seed=seed)
    loss = reference_main_loss(out)
    loss.backward()
    opt.step()
    return float(loss)


def build_oracle(levels):
    from oracle import lidar4d_oracle as O
    from lidar4d_b200.geometry import FieldConfig
    cfg = FieldConfig(**model_kwargs(levels))
    torch.manual_seed(0)
    orc = O.OracleLiDAR4D(cfg)
    O.randomize_parameters(orc, seed=0, flow_last_std=1e-3)
    opt = torch.optim.Adam(orc.parameters(), lr=1e-2, betas=(0.9, 0.99), eps=1e-15)
    return orc, opt


def cpu_sample(levels, n_rays, repeats=1):
    """rays/s of the oracle on this box's host cores for a bounded sample of the workload."""
    from lidar4d_b200.rays import synthetic_sweep
    orc, opt = build_oracle(levels)
    ro, rd, t = synthetic_sweep(7, N_FRAMES, H_SWEEP, W_SWEEP)
    sel = np.linspace(0, ro.shape[0] - 1, n_rays).astype(np.int64)
    cpu_reference_step(orc, opt, ro[sel], rd[sel], float(t), 0)         # warm-up
    ts = []
    for i in range(repeats):
        t0 = time.perf_counter()
        cpu_reference_step(orc, opt, ro[sel], rd[sel], float(t), i + 1)
        ts.append(time.perf_counter() - t0)
    dt = float(np.median(ts))
    return n_rays / dt, dt


def cpu_threads():
    """Threads for the CPU arm: every core up to 32 (the oracle's index/scatter ops stop scaling there and
    oversubscribed boxes get slower, not faster)."""
    return max(1, min(32, os.cpu_count() or 1))


def cpu_baseline_subprocess(args):
    """Time the oracle port in a child process (bounded by a wall-clock guard so the bench always finishes)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1",
           "--cpu-rays", str(args.cpu_rays), "--levels", str(args.levels)]
    log("cpu_baseline: " + " ".join(cmd[2:]))
    try:
        env = dict(os.environ, RANK="0", WORLD_SIZE="1", CUDA_VISIBLE_DEVICES="")
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=420, env=env)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"value": None, "unit": "rays/s", "cores": cpu_threads(), "kind": "port", "sample": "failed: " + r.stderr[-200:]}
    except subprocess.TimeoutExpired:
        return {"value": None, "unit": "rays/s", "cores": cpu_threads(), "kind": "port",
                "sample": f"{args.cpu_rays} rays did not finish in 420 s"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; tiny-cuda-nn is absent)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(cpu_threads())
    from lidar4d_b200.rays import synthetic_sweep
    log(f"reference arm: oracle port on {torch.get_num_threads()} host threads, L={args.levels}")
    orc, opt = build_oracle(args.levels)
    n = args.cpu_rays
    ts = []
    for i in range(args.warmup + args.steps):
        ro, rd, t = synthetic_sweep(i % N_FRAMES, N_FRAMES, H_SWEEP, W_SWEEP)
        sel = np.linspace(0, ro.shape[0] - 1, n).astype(np.int64)
        t0 = time.perf_counter()
        cpu_reference_step(orc, opt, ro[sel], rd[sel], float(t), i)
        log(f"reference step {i}: {time.perf_counter() - t0:.2f} s")
        if i >= args.warmup:
            ts.append(time.perf_counter() - t0)
    total = float(sum(ts))
    val = n * args.steps / total
    sample = f"{n} rays x {S_STEPS} samples fwd+bwd+Adam per step (bounded sample of the 65,536-ray sweep), fp32"
    line = {
        "impl": "reference", "metric": "training rays/sec at 64x1024 rays x 768 samples", "value": val, "unit": "rays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, note="CPU: oracle port of the reference python path on the tcnn spec"),
        "cpu_baseline": {"value": val, "unit": "rays/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, note=None):
    c = {"workload": f"synthetic KITTI-360-like sweep {H_SWEEP}x{W_SWEEP} rays x {S_STEPS} samples, "
                     f"L={args.levels} 4D hash (2^19 static, 2^15/2^13/2^13 x8 time slices) + 6 hex-planes x4 scales + flow field, "
                     f"{N_FRAMES} frames",
         "rays_per_step": args.rays, "ray_batch": args.ray_batch, "n_levels_hash": args.levels,
         "parallelism": f"ray-sharded dp{args.gpus}", "streams": getattr(args, "streams", 1), "loss": getattr(args, "loss", None), "pipeline": getattr(args, "pipeline", None), "mlp": getattr(args, "mlp", None),
         "l2": "inputs larger than L2: fp16/fp32 working set > 126 MB plus > 1 GB of saved activations streamed per step"}
    if note:
        c["note"] = note
    return c


# =============================================================================
# GPU arm
# =============================================================================
STATIC_AGG_RES = 1200        # L4D_STATIC_AGG_RES of lidar4d_b200/csrc/l4d_split.cuh (levels whose runs of equal cells are summed in the warp)


def red_counts(cfg, rays=None):
    """Vector reductions (RED.E.ADD.F32x4 lane-ops) per sample that k_bwd_scatter_static EXECUTES - the kernel whose ceiling is
    the L2 atomic unit (DESIGN.md 4.2 'atomic floor').  Algorithmically it is one per hash corner (8 L); at the levels up to
    res 1200 the kernel sums every run of consecutive samples of a warp that share their cell and issues the 8 corners once per
    run, so the executed count is 8 x runs / samples there: the run statistics are computed here, on the host, from the
    benchmark's own rays (unjittered z grid), the same way the kernel forms its runs (32 consecutive samples of a ray)."""
    L = cfg.n_levels_hash
    g = cfg.static_grid()
    out = {"k_bwd_scatter_static": float(L * 8), "k_bwd_scatter_static_algorithmic": float(L * 8)}
    if rays is None:
        return out
    ro, rd = rays
    ro, rd = np.asarray(ro, np.float32)[:256], np.asarray(rd, np.float32)[:256]
    z = np.linspace(np.float32(cfg.near_lidar), np.float32(cfg.far_lidar), S_STEPS, dtype=np.float32)
    x01 = (ro[:, None, :] + rd[:, None, :] * z[None, :, None] + np.float32(cfg.bound)) / np.float32(2 * cfg.bound)   # [rays, S, 3]
    executed = 0.0
    for l in range(L):
        if int(g.resolution[l]) > STATIC_AGG_RES:
            executed += 8.0
            continue
        cell = np.floor(x01 * g.scale[l] + np.float32(0.5)).astype(np.int64)
        key = cell[..., 0] + int(g.resolution[l]) * (cell[..., 1] + int(g.resolution[l]) * cell[..., 2])      # [rays, S]
        key = key.reshape(key.shape[0], -1, 32)                      # warps of 32 consecutive samples (S is a multiple of 32)
        runs = 1 + (key[..., 1:] != key[..., :-1]).sum(-1)           # runs per warp
        executed += 8.0 * float(runs.sum()) / float(key.size)
    out["k_bwd_scatter_static"] = executed
    return out


def micro_peaks():
    """Measured ceilings of the units that actually bind the kernels (profiles/r02_micro_peaks.json, from
    scripts/micro/{gather,red}_bench.cu on a B200 of this pool): divergent L2-resident sector gathers, RED.128 lane-ops."""
    p = os.path.join(ROOT, "profiles", "r02_micro_peaks.json")
    if os.path.exists(p):
        return json.load(open(p))
    return {}


def ncu_binding():
    p = os.path.join(ROOT, "profiles", "ncu_binding.json")
    return json.load(open(p)) if os.path.exists(p) else {}


DUMP_SAMPLE = 1 << 16        # --dump-outputs: entries kept of each parameter tensor larger than this


def dump_outputs(out_dir, model, last, with_params):
    """--dump-outputs: the arrays the last timed step handed its caller, as float32 / float64 .npy files (about 20 MB at
    the default workload): depth [rays], image [rays, 2], loss [1] and, after a training step, grad_sample / param_sample,
    the gradients and updated parameters of every tensor in named_parameters() order.  A tensor larger than DUMP_SAMPLE
    contributes the entries at a seeded random set of DUMP_SAMPLE positions, the same set on every run."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"depth": torch.cat([d.reshape(-1) for d, _ in last["chunks"]]),
              "image": torch.cat([i.reshape(-1, 2) for _, i in last["chunks"]])}
    if "loss" in last:
        arrays["loss"] = last["loss"].double().reshape(1)
    if with_params:
        grads, params = [], []
        for k, p in enumerate(model.parameters()):
            flat = p.detach().reshape(-1)
            g = p.grad.reshape(-1) if p.grad is not None else torch.zeros_like(flat)
            if flat.numel() > DUMP_SAMPLE:
                pos = np.sort(np.random.default_rng(k).choice(flat.numel(), DUMP_SAMPLE, replace=False))
                pos = torch.from_numpy(pos).to(flat.device)
                flat, g = flat[pos], g[pos]
            params.append(flat.float())
            grads.append(g.float())
        arrays["grad_sample"], arrays["param_sample"] = torch.cat(grads), torch.cat(params)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().cpu().numpy())
    log(f"outputs of the last timed step: {', '.join(f'{n} {tuple(a.shape)}' for n, a in arrays.items())} -> {out_dir}")


def gpu_eager_baseline(levels, n_rays, dev):
    """SURVEY.md 8(d)(ii) / BASELINE.md 3 'B-gpu-eager': the reference's op graph (the oracle = its plain-torch restatement,
    pinned to the reference modules to 1e-6; the modules themselves live in /root/reference, which does not exist on the GPU
    box) executed eagerly on THIS GPU under fp16 autocast as runner.py:497 does, fwd + bwd + Adam, bounded sample.
    A baseline leg like cpu_baseline: the only thing here that touches oracle/ on a GPU."""
    from lidar4d_b200.rays import synthetic_sweep
    try:
        orc, _ = build_oracle(levels)
        orc = orc.to(dev)
        opt = torch.optim.Adam(orc.parameters(), lr=1e-2, betas=(0.9, 0.99), eps=1e-15)
        scaler = torch.amp.GradScaler("cuda")
        ro, rd, t = synthetic_sweep(7, N_FRAMES, H_SWEEP, W_SWEEP)
        sel = np.linspace(0, ro.shape[0] - 1, n_rays).astype(np.int64)
        ro_t, rd_t = torch.from_numpy(ro[sel]).to(dev), torch.from_numpy(rd[sel]).to(dev)

        def one(seed):
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.float16):
                out = orc.render(ro_t, rd_t, float(t), num_steps=S_STEPS, perturb=True, seed=seed)
                loss = reference_main_loss(out)
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        for i in range(2):
            one(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        torch.cuda.reset_peak_memory_stats()
        e0.record()
        for i in range(reps):
            one(10 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res = {"value": n_rays / (ms * 1e-3), "unit": "rays/s", "ms_per_step": ms, "rays_per_step": n_rays,
               "peak_mem_gb": torch.cuda.max_memory_allocated() / 1e9, "kind": "port",
               "what": "oracle (plain-torch restatement of the reference op graph on the tcnn spec) in GPU eager mode, fp16 autocast + "
                       "GradScaler, fwd+bwd+Adam; tiny-cuda-nn itself cannot be built here"}
        del orc, opt
        torch.cuda.empty_cache()
        return res
    except Exception as e:          # a baseline leg must never take the bench line down
        return {"value": None, "unit": "rays/s", "error": repr(e)[:200]}


def run_b200(args):
    import torch.distributed as dist
    from lidar4d_b200 import LiDAR4D
    from lidar4d_b200.rays import synthetic_sweep
    from lidar4d_b200.parallel import RayShardedDP, shard_range
    from lidar4d_b200.optim import Adam          # main_lidar4d.py:298-300 recipe, one launch fused with the fp16 table refresh

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    infer = args.mode == "infer"
    if infer and args.rays == H_SWEEP * W_SWEEP:
        args.rays = 64 * 2048                        # BASELINE.json configs[3]
    strong = args.scaling == "strong" and not infer

    torch.manual_seed(0)
    model = LiDAR4D(**model_kwargs(args.levels)).to(dev)
    randomize(model, 0)
    model.materialize_weights = False            # weights/z_vals are only read by --urf_loss (runner.py:256-276)
    model.pipeline = args.pipeline
    model.set_mlp_fp16(args.mlp == "fp16")
    dp = RayShardedDP(model, world_size=world, rank=rank)
    opt = Adam(model, model.get_params(1e-2), betas=(0.9, 0.99), eps=1e-15)
    rb = args.ray_batch
    # rays of this rank per step: weak = a whole sweep each, strong = a contiguous 1/R shard of the global batch
    lo, hi = shard_range(args.rays, world, rank) if strong else (0, args.rays)
    n_rays = hi - lo
    global_rays = args.rays if strong else args.rays * world
    W_frame = 2048 if infer else W_SWEEP

    # host-side inputs in pinned memory (one sweep per frame)
    frames = []
    for k in range(min(N_FRAMES, args.warmup + args.steps + 1)):
        fid = (k if strong else k * world + rank) % N_FRAMES
        ro, rd, t = synthetic_sweep(fid, N_FRAMES, H_SWEEP, W_frame)
        if args.rays < ro.shape[0]:
            # a batch smaller than the sweep is a RANDOM pixel subset, as the reference's loader draws it
            # (base_dataset.py:71 torch.randint over H*W; kitti360_dataset.py:159-166) - not the first rows of the sweep,
            # whose rays share one elevation and pile their plane-gradient reductions onto a few texels
            sel = np.random.default_rng(1000 + fid).permutation(ro.shape[0])[:args.rays]
            ro, rd = ro[sel], rd[sel]
        ro, rd = ro[lo:hi] if strong else ro[:n_rays], rd[lo:hi] if strong else rd[:n_rays]
        frames.append((torch.from_numpy(np.ascontiguousarray(ro)).pin_memory(), torch.from_numpy(np.ascontiguousarray(rd)).pin_memory(), float(t)))
    host_out = torch.empty(n_rays, 3).pin_memory()
    from lidar4d_b200.losses import lidar_main_loss
    gt_d = torch.tensor([1.0, 0.5, 0.3], device=dev).repeat(n_rays, 1)      # (no drop, intensity 0.5, depth 0.3) for every ray
    ray_off0 = lo if strong else rank * n_rays

    def inputs(i, e2e):
        ro_h, rd_h, t = frames[i % len(frames)]
        if e2e:
            return ro_h.to(dev, non_blocking=True), rd_h.to(dev, non_blocking=True), t
        if getattr(inputs, "resident", None) is None or inputs.resident[0] != i % len(frames):
            inputs.resident = (i % len(frames), ro_h.to(dev), rd_h.to(dev))
        return inputs.resident[1], inputs.resident[2], t

    n_chunks = (n_rays + rb - 1) // rb
    n_streams = max(1, min(args.streams, n_chunks))
    side = [torch.cuda.Stream(device=dev) for _ in range(n_streams)] if n_streams > 1 else []

    latest = {}         # --dump-outputs: the outputs of the step that ran last (references only: no work on the device)

    def chunk(h, ro_d, rd_d, t, e2e, last):
        out = model.render(ro_d[None, h:h + rb], rd_d[None, h:h + rb], t, staged=False, num_steps=S_STEPS,
                           perturb=True, ray_offset=ray_off0 + h)
        if args.dump_outputs:
            latest["chunks"].append((out["depth_lidar"].detach(), out["image_lidar"].detach()))
        # the reference's main loss (runner.py:193-213: L1 depth, label-smoothed ray-drop MSE, intensity MSE, defaults of
        # main_lidar4d.py:70-72,88) against a synthetic ground-truth image, value + gradient in one launch
        if args.loss == "unit":       # round 1's synthetic loss (unit weights): kept as the default so that rounds compare like for like
            loss = ((out["depth_lidar"] - 0.3).abs().sum() + ((out["image_lidar"] - 0.5) ** 2).sum()) / global_rays
        else:                         # the reference's main loss and weights (runner.py:193-213) in one launch, value + gradient
            loss = lidar_main_loss(out["depth_lidar"], out["image_lidar"], gt_d[None, h:h + rb], 1.0, 0.01, 0.1, 0.2) * (1.0 / global_rays)
        if last:
            dp.final_backward(loss)          # the hash-table bucket starts reducing while the flow backward still runs
        else:
            loss.backward()
        res = None
        if e2e:
            res = torch.cat([out["depth_lidar"].detach().view(-1, 1), out["image_lidar"].detach().view(-1, 2)], 1)
        return loss.detach(), res

    def train_step(i, e2e, streams=True):
        ro_d, rd_d, t = inputs(i, e2e)
        latest.clear()
        latest["chunks"] = []
        opt.zero_grad(set_to_none=True)
        main = torch.cuda.current_stream()
        parts, outs = [], []
        if side and streams:
            model.prepare_grads()             # attach + clear the gradient arena once, before the streams fork
            for st in side:
                st.wait_stream(main)
            for c, h in enumerate(range(0, n_rays, rb)):
                with torch.cuda.stream(side[c % n_streams]):
                    l, r = chunk(h, ro_d, rd_d, t, e2e, False)
                    parts.append(l)
                    outs.append(r)
            for st in side:
                main.wait_stream(st)
            for x in parts + [r for r in outs if r is not None]:
                x.record_stream(main)
        else:
            for h in range(0, n_rays, rb):
                l, r = chunk(h, ro_d, rd_d, t, e2e, h + rb >= n_rays)
                parts.append(l)
                outs.append(r)
        tot = torch.stack(parts).sum()
        latest["loss"] = tot
        dp.allreduce_grads()
        if train_step.adam_events is not None:        # profile pass: time the fused Adam + staging launch pair
            ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
            ev[0].record()
            opt.step()
            ev[1].record()
            train_step.adam_events.append(ev)
        else:
            opt.step()
        if e2e:
            host_out.copy_(torch.cat(outs, 0), non_blocking=True)
            return float(tot)            # device->host read of the step's loss (sync)
        return tot

    train_step.adam_events = None

    def infer_step(i, e2e):
        ro_d, rd_d, t = inputs(i, e2e)
        with torch.no_grad():
            out = model.render(ro_d[None], rd_d[None], t, staged=False, num_steps=S_STEPS, perturb=False, ray_offset=ray_off0)
        latest.clear()
        latest["chunks"] = [(out["depth_lidar"], out["image_lidar"])]
        if e2e:
            host_out[:, 0:1].copy_(out["depth_lidar"].view(-1, 1), non_blocking=True)
            host_out[:, 1:3].copy_(out["image_lidar"].view(-1, 2), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return out["depth_lidar"]

    step = infer_step if infer else train_step
    if infer:
        model.eval()
        model.static_params(True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(e2e, n_steps, base):
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = model.gpu_launches
        ev0.record()
        for i in range(n_steps):
            step(base + i, e2e)
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1:
            tm = torch.tensor([ms], device=dev)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            ms = float(tm)
        return ms, model.gpu_launches - l0

    log(f"model ready (L={args.levels}), mode {args.mode}, {args.scaling} scaling: {n_rays} rays/step on this rank in launches of {rb}")
    for i in range(args.warmup):
        tw = time.perf_counter()
        step(i, False)
        torch.cuda.synchronize()
        log(f"warm-up step {i}: {time.perf_counter() - tw:.2f} s")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, launches = timed(False, args.steps, args.warmup)
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, latest, with_params=not infer)
    log(f"timed: {ms / args.steps:.2f} ms/step")
    step(0, True)                                  # warm the e2e path (pinned copies)
    ms_e2e, _ = timed(True, args.steps, args.warmup)
    peak_mem = torch.cuda.max_memory_allocated() / 1e9

    # ---- per-kernel durations for the roofline: CUDA events recorded by the library on the launch stream ----
    from lidar4d_b200 import _capi
    torch.cuda.synchronize()
    # (serial: the library's event marks time one stream)
    train_step.adam_events = []
    ktimes = _capi.profile_kernels(lambda: [(train_step(args.warmup + i, False, streams=False) if not infer else step(args.warmup + i, False)) for i in range(2)])
    torch.cuda.synchronize()
    if train_step.adam_events:
        ktimes["k_adam_flat+k_stage_jobs"] = [a.elapsed_time(b) for a, b in train_step.adam_events]
    train_step.adam_events = None

    regimes = None
    if not infer:
        # ---- SURVEY 8(d): the two density regimes and their measured attribute-mask fraction M/P ----
        def mask_fraction():
            keep = model.materialize_weights
            model.materialize_weights = True
            with torch.no_grad():
                ro_h, rd_h, t = frames[0]
                sel = torch.linspace(0, n_rays - 1, min(1024, n_rays)).long()
                out = model.render(ro_h[sel].to(dev)[None], rd_h[sel].to(dev)[None], t, staged=False, num_steps=S_STEPS, perturb=False)
                mf = float((out["weights"] > 1e-4).float().mean())
            model.materialize_weights = keep
            return mf

        regimes = {"init-like": {"mask_fraction": mask_fraction(), "rays_per_s": global_rays * args.steps / (ms * 1e-3)}}
        with torch.no_grad():           # surface-like: positive, scaled sigma row => the weight mass sits in a few samples per ray
            pz = model.sigma_net.params
            off = 64 * model.cfg.sigma_in_pad
            pz[off:off + 64] = pz[off:off + 64].abs() * 4.0
        step(0, False)
        ms_s, _ = timed(False, 2, 1)
        regimes["surface-like"] = {"mask_fraction": mask_fraction(), "rays_per_s": global_rays * 2 / (ms_s * 1e-3)}
        log(f"regimes: {regimes}")

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    samples_per_launch = min(rb, n_rays) * S_STEPS if not infer else min(model.infer_ray_chunk, n_rays) * S_STEPS
    kbytes = kernel_bytes(model.cfg)
    reds = red_counts(model.cfg, (frames[0][0].numpy(), frames[0][1].numpy()) if S_STEPS % 32 == 0 else None)
    mp = micro_peaks()
    nb = ncu_binding()
    nbk = nb.get("kernels", {})
    kern = {}
    for name, ts in ktimes.items():
        avg = float(np.mean(ts))
        b = kbytes.get(name.replace("_tc", ""), None)
        k = {"avg_ms": avg, "launches_timed": len(ts), "alg_bytes_per_sample": b,
             "alg_gbs_l2_resident_not_a_dram_bound": (b * samples_per_launch / (avg * 1e-3) / 1e9) if b else None}
        if name in reds and mp.get("red128_glaneops_s"):
            rate = reds[name] * samples_per_launch / (avg * 1e-3) / 1e9
            k["binding"] = {"unit": "L2 atomic unit: G RED.128 lane-ops/s", "achieved": rate, "peak": mp["red128_glaneops_s"],
                            "frac": rate / mp["red128_glaneops_s"], "red_lane_ops_per_sample_executed": reds[name],
                            "red_lane_ops_per_sample_algorithmic": reds.get(name + "_algorithmic"),
                            "source": "live duration x executed REDs (8 per level, 8 x runs/samples at the warp-aggregated levels: host-side run "
                                      "statistics of the benchmark's rays) vs scripts/micro/red_bench.cu (profiles/r02_micro_peaks.json)"}
        elif name in nb.get("stale", {}):
            # the committed ncu capture predates this kernel's current code: name the unit it was bound by then, claim no fraction
            k["binding"] = {"unit": nbk.get(name, {}).get("limiter_unit"), "frac": None, "achieved": None, "peak": None,
                            "stale": nb["stale"][name], "last_capture": nbk.get(name, {}).get("limiter")}
        elif name in nbk and nbk[name].get("limiter_pct") is not None:
            k["binding"] = {"unit": nbk[name]["limiter_unit"], "frac": nbk[name]["limiter_pct"] / 100.0,
                            "achieved": nbk[name]["limiter_pct"], "peak": 100.0, "achieved_unit": "% of the unit's peak rate (ncu)",
                            "source": f"ncu --set full capture of this kernel ({nb.get('source')}): the profiler's own achieved/peak ratio of the busiest unit"}
        if name in nbk and name not in nb.get("stale", {}):
            k["ncu"] = nbk[name]
        kern[name] = k
    dom = max(kern, key=lambda k: kern[k]["avg_ms"]) if kern else None
    traffic = None
    try:        # dram__bytes_read+write of the dominant kernel from the committed ncu capture (scaled to this launch size)
        tj = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        if args.levels == 16 and tj["dram_bytes_per_launch"].get(dom) is not None and dom not in nb.get("stale", {}):
            traffic = tj["dram_bytes_per_launch"][dom] * (samples_per_launch / (float(tj.get("rays_per_launch", 8192)) * S_STEPS))
    except Exception:
        traffic = None
    roofline = None
    if dom:
        kd = kern[dom]
        bind = kd.get("binding") or {}
        alg = kd["alg_gbs_l2_resident_not_a_dram_bound"]
        dram_gbs = (traffic / (kd["avg_ms"] * 1e-3) / 1e9) if traffic else None
        # `bound` names the unit that binds the dominant kernel and `frac` is achieved/peak of THAT unit; the HBM view
        # (measured DRAM bytes and the algorithmic-bytes figure of SURVEY 8(d)) sits beside it under "hbm"
        roofline = {"bound": bind.get("unit", "hbm"), "kernel": dom, "achieved": bind.get("achieved"), "peak": bind.get("peak"),
                    "unit": bind.get("achieved_unit", "G lane-ops/s"),
                    "frac": bind.get("frac"), "traffic": traffic, "source": bind.get("source"),
                    "hbm": {"bound": "hbm", "measured_dram_gbs": dram_gbs, "peak": peak, "unit": "GB/s",
                            "frac": (dram_gbs / peak) if dram_gbs else None, "peak_source": peak_src, "algorithmic_gbs": alg,
                            "note": "algorithmic bytes (SURVEY 8(d)) / duration: the fp16 tables and the live gradient slabs are L2-resident, "
                                    "so this is NOT a DRAM bound and may exceed the HBM peak; measured_dram_gbs = ncu dram bytes / live duration"},
                    "kernels": kern}
    total_rays = global_rays * args.steps
    value = total_rays / (ms * 1e-3)
    metric = ("inference rays/sec at 64x2048 rays x 768 samples" if infer else "training rays/sec at 64x1024 rays x 768 samples")
    cfgd = workload_config(args)
    cfgd.update({"rays_per_step": global_rays, "rays_per_rank": n_rays, "mode": args.mode,
                 "optimizer": "lidar4d_b200.optim.Adam (one launch, fused fp16 table refresh)" if not infer else None})
    line = {
        "metric": metric, "value": value, "unit": "rays/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": ("fp16 tables + fp16 MLP weights (tcgen05, hi/lo fp16 activations, fp32 accumulate)" if args.mlp == "fp16"
                  else "fp16 tables, fp32 MLPs") + "; fp32 planes, compositing and gradients", "data": "synthetic",
        "config": cfgd,
        "e2e": {"value": total_rays / (ms_e2e * 1e-3), "unit": "rays/s", "h2d_bytes_per_step": n_rays * 6 * 4,
                "d2h_bytes_per_step": n_rays * 3 * 4 + (0 if infer else 4), "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "regimes": regimes, "peak_mem_gb": peak_mem,
    }
    log(f"e2e {ms_e2e / args.steps:.2f} ms/step; kernels " + ", ".join(f"{k} {v['avg_ms']:.2f} ms" for k, v in kern.items()))
    if world == 1 and not infer:
        if args.eager_rays > 0:
            torch.cuda.empty_cache()
            line["gpu_eager_baseline"] = gpu_eager_baseline(args.levels, args.eager_rays, dev)
            log(f"gpu_eager_baseline: {line['gpu_eager_baseline']}")
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_subprocess(args)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)
