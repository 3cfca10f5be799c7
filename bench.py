#!/usr/bin/env python
"""bench.py -- transition frames/sec of the branch-tree denoising hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4|5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one ``BlendingEngine.run_transition()`` of the selected BASELINE.json config (default: configs[1], the
one the metric is quoted on): SDXL-base-shaped UNet (2.57 B random-init parameters), 1024x1024 (128x128 latents),
30 Euler steps, depth_strength 0.5, nmb_max_branches 15 -> 15 frames, 198 CFG-batch-2 UNet forwards, 13 parental
mixes, 15 VAE decodes, 26 LPIPS evaluations.  ``--config 3`` = 30 branches with parental + branch-1 crossfeed
(0.8/0.6/0.4, README.md:122), ``--config 5`` = SDXL-Turbo 512x512, 4 steps, 60 branches, ``--config 4`` = the
8-prompt multi-transition loop of example_multi_trans.py (7 transitions per step, time-based branching).
Synthetic data (no network): seeded random weights / embeddings, fixed seeds.

Prints ONE JSON line (rank 0).  ``value`` = frames/s with the conditioning already on the device and frames left on
the device; ``e2e`` = the same through the public API (set_prompt1/2 -> run_transition -> PIL frames), host<->device
copies timed.  ``fingerprint`` = sha1 over the tree (tree_fracts, tree_idx_injection, every branch's final latents):
equal fingerprints across --gpus 1/2/4/8 mean the sharded run built exactly the single-GPU tree.
``--dump-outputs DIR`` writes the frames, final latents and fractions of the last timed step as .npy files, so that
two builds can be compared output for output on the same seeded inputs.
``--impl reference`` times the CPU oracle (a port of the reference path: diffusers / lpips are not installable
here) on the host cores this process may use.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PROMPTS = ("photo of underwater landscape, fish, und the sea, incredible detail, high resolution",
           "rendering of an alien planet, strange plants, strange creatures, surreal")
PROMPTS_MULTI = ("high resolution ultra 8K image with lake and forest", "strange and alien desolate lanscapes 8K",
                 "ultra high res psychedelic skyscraper city landscape 8K unreal engine",
                 "photo of a quiet harbour at dawn, fishing boats, mist", "macro photo of frost crystals on a leaf",
                 "wide desert canyon under a storm, dramatic light", "dense jungle waterfall, volumetric light",
                 "aerial photo of terraced rice fields at sunset")
NEG = "blurry, ugly, pale"
L2_NOTE = "working set (5.1 GB fp16 weights per UNet forward) exceeds L2; no flush needed"

CONFIGS = {
    2: dict(metric="transition frames/sec (1024^2 SDXL, 30 steps, 15 branches)", model="base", latent=128,
            num_inference_steps=30, depth_strength=0.5, nmb_max_branches=15, branch1_crossfeed=None,
            stems=[4, 3, 3, 2, 1], frames=15, unet_forwards=198, cfg_batch=2, mixes=13, lpips=26, seeds=[420, 421],
            workload="single_trans SDXL 1024x1024, 30 steps, depth_strength=0.5, nmb_max_branches=15"),
    3: dict(metric="transition frames/sec (1024^2 SDXL, 30 steps, 30 branches, parental+branch1 crossfeed)",
            model="base", latent=128, num_inference_steps=30, depth_strength=0.5, nmb_max_branches=30,
            branch1_crossfeed=(0.8, 0.6, 0.4), stems=[7, 6, 6, 5, 4], frames=30, unet_forwards=333, cfg_batch=2,
            mixes=28, lpips=56, seeds=[420, 421],
            workload="single_trans SDXL 1024x1024, 30 steps, nmb_max_branches=30, parental (0.3/0.6/0.9) + branch1 "
                     "(0.8/0.6/0.4) crossfeed"),
    4: dict(metric="multi-transition frames/sec (8 prompts, 1024^2 SDXL, 30 steps, t_compute_max_allowed)",
            model="base", latent=128, num_inference_steps=30, depth_strength=0.5, nmb_max_branches=None,
            branch1_crossfeed=None, stems=None, frames=None, unet_forwards=None, cfg_batch=2, seeds="420+i",
            workload="multi_trans 8 prompts SDXL 1024x1024, 30 steps, time-based branching, 7 transitions "
                     "(6 recycle keyframe 1 via swap_forward)"),
    5: dict(metric="transition frames/sec (512^2 SDXL-Turbo, 4 steps, 60 branches)", model="turbo", latent=64,
            num_inference_steps=4, depth_strength=None, nmb_max_branches=60, branch1_crossfeed=None, stems=[60],
            frames=62, unet_forwards=128, cfg_batch=1, mixes=60, lpips=120, seeds=[420, 421],
            workload="single_trans SDXL-Turbo 512x512, 4 steps, nmb_max_branches=60"),
}


def peaks():
    p = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")
    fp = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(fp):
        with open(fp) as f:
            p.update(json.load(f))
        p["source"] = "measured"
    return p


def measured_traffic():
    """dram__bytes_read+write per launch from the committed ncu capture (profiles/traffic.json, written by
    tools/ncu_traffic.py from an `ncu --metrics dram__bytes_*` pass over one UNet forward / one batched mix)."""
    fp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(fp):
        with open(fp) as f:
            return json.load(f)
    return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        self.th.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores
# Analytic FLOPs of one SDXL UNet sample (SURVEY.md section 8d): everything but self-attention scales with the
# number of latent pixels, self-attention QK^T / PV with its square.
_UNET_TFLOP_1024 = dict(linear_conv=5.977, self_attn=0.752, cross_attn=0.032)


def unet_tflop(latent):
    r = (latent / 128.0) ** 2
    u = _UNET_TFLOP_1024
    return (u["linear_conv"] + u["cross_attn"]) * r + u["self_attn"] * r * r


def host_cpu_budget():
    """CPUs this process may actually use: scheduler affinity capped by the cgroup CPU quota (v2 cpu.max or v1
    cfs_quota).  os.cpu_count() reports the whole host, which oversubscribes a 1-GPU slice of a shared box."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
        if q != "max":
            quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f:
                q = float(f.read())
            with open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as f:
                p = float(f.read())
            if q > 0:
                quota = q / p
        except Exception:
            pass
    if quota is not None:
        n = min(n, max(1, int(quota + 0.5)))
    return max(1, n)


def pick_threads():
    """Thread count for the CPU arm: start from the affinity / cgroup budget, then MEASURE a fp32 GEMM with that count
    and its halves and keep the fastest -- a shared host can be busier than its limits say.  Returns (threads,
    gflops, detail)."""
    import torch
    budget = host_cpu_budget()
    cands, c = [], budget
    while c >= 1 and len(cands) < 5:
        cands.append(c)
        c //= 2
    a = torch.randn(2048, 2048)
    b = torch.randn(2048, 2048)
    flop = 2.0 * 2048 ** 3
    detail, best = {}, (0.0, 1)
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.time()
        reps = 0
        while reps < 3 or (time.time() - t0 < 0.3 and reps < 20):
            a @ b
            reps += 1
        gf = flop * reps / (time.time() - t0) / 1e9
        detail[str(c)] = round(gf, 1)
        if gf > best[0] * 1.05:         # prefer more threads only when they pay
            best = (gf, c)
        if gf < 0.5 * best[0]:
            break
    torch.set_num_threads(best[1])
    return best[1], best[0], dict(budget=budget, os_cpu_count=os.cpu_count(), gemm_gflops_by_threads=detail)


class CpuPort:
    """Bounded sample of the CPU oracle for one config.  HEAVY legs (one fp32 UNet forward at the config's CFG batch,
    one VAE decode) run ONCE -- at the config's full latent size when the measured GEMM rate predicts <= 75 s for the
    UNet forward, else at the largest halved size that does; LIGHT legs (one full-size parental mix, one LPIPS pair at the sample size) run every step.  Times
    are scaled to the config's shape by the analytic FLOP / pixel ratios and the transition time is extrapolated with
    the config's exact call counts (SURVEY.md section 8d).  A full-size CPU transition would take hours."""

    def __init__(self, cfg):
        import torch
        self.cfg = cfg
        self.threads, self.gemm_gflops, self.thread_detail = pick_threads()
        L_full = cfg["latent"]
        B = cfg["cfg_batch"]
        # predicted seconds of the heavy UNet sample at ~70 % of the GEMM rate
        self.L = L_full
        while self.L > 16 and B * unet_tflop(self.L) * 1e3 / (0.7 * max(self.gemm_gflops, 1.0)) > 75.0:
            self.L //= 2
        self.heavy = None
        self.torch = torch

    def _build(self):
        torch = self.torch
        from oracle.lpips_alex import LPIPSAlex
        from oracle.sdxl_unet import SDXL_BASE, SDXLUNet
        from oracle.vae import SDXL_VAE, VAEDecoder
        t0 = time.time()
        with torch.no_grad():
            # timing only: parameters are filled with small uniform noise (the default nn inits of 2.57 B parameters
            # cost minutes of single-threaded RNG; the arithmetic does not depend on the values)
            with torch.device("meta"):
                unet = SDXLUNet(SDXL_BASE)
            unet = unet.to_empty(device="cpu").eval()
            for p in unet.parameters():
                p.uniform_(-0.02, 0.02)
            self.unet = unet
            self.vae = VAEDecoder(SDXL_VAE).eval()
            self.lpips = LPIPSAlex()
        g = torch.Generator().manual_seed(0)
        L, B = self.L, self.cfg["cfg_batch"]
        self.x = torch.randn(B, 4, L, L, generator=g)
        self.ctx = torch.randn(B, 77, 2048, generator=g) * 0.5
        self.pool = torch.randn(B, 1280, generator=g)
        self.tid = torch.tensor([[8. * L, 8. * L, 0, 0, 8. * L, 8. * L]] * B)
        self.lat = torch.randn(1, 4, L, L, generator=g).half()
        Lf, N = self.cfg["latent"], self.cfg["num_inference_steps"]
        self.traj = [torch.randn(1, 4, Lf, Lf, generator=g).half() for _ in range(2 * N)]
        self.t_build = time.time() - t0

    def step(self):
        """One bench step of the CPU arm -> dict of timings + extrapolated frames/s."""
        torch = self.torch
        from oracle import mixing
        from oracle.lpips_alex import lpips_distance
        from oracle.vae import latent2image_np
        if self.heavy is None:
            self._build()
            with torch.no_grad():
                t0 = time.time()
                self.unet(self.x, 500.0, self.ctx, self.pool, self.tid)
                t_unet = time.time() - t0
                t0 = time.time()
                self.img = latent2image_np(self.vae, self.lat)
                t_vae = time.time() - t0
            self.heavy = dict(t_unet_sample=t_unet, t_vae_sample=t_vae)
        N = self.cfg["num_inference_steps"]
        with torch.no_grad():
            t0 = time.time()
            mixing.parental_mix(self.traj[:N], self.traj[N:], 0.4)
            t_mix = time.time() - t0
            t0 = time.time()
            lpips_distance(self.lpips, self.img, self.img[::-1].copy())
            t_lpips_s = time.time() - t0
        c, L, Lf, B = self.cfg, self.L, self.cfg["latent"], self.cfg["cfg_batch"]
        px = (float(Lf) / L) ** 2
        t_unet = self.heavy["t_unet_sample"] * unet_tflop(Lf) / unet_tflop(L)
        t_vae = self.heavy["t_vae_sample"] * px
        t_lpips = t_lpips_s * px
        frames, fw = c["frames"] or 15, c["unet_forwards"] or 198
        mixes, lp = c.get("mixes") or 13, c.get("lpips") or 26
        total = fw * t_unet + frames * t_vae + mixes * t_mix + lp * t_lpips
        return dict(frames_per_s=frames / total, transition_s_extrapolated=total, t_unet_fwd=t_unet, t_vae=t_vae,
                    t_mix=t_mix, t_lpips=t_lpips, t_unet_fwd_sample=self.heavy["t_unet_sample"],
                    t_vae_sample=self.heavy["t_vae_sample"], t_lpips_sample=t_lpips_s,
                    unet_sample_gflops=B * unet_tflop(L) * 1e3 / self.heavy["t_unet_sample"])

    def sample_text(self):
        c, L, Lf = self.cfg, self.L, self.cfg["latent"]
        return (f"bounded sample on {self.threads} host threads (fp32 GEMM probe {self.gemm_gflops:.0f} GFLOP/s): ONE fp32 "
                f"CFG-batch-{c['cfg_batch']} SDXL UNet forward (2.57 B params) and ONE VAE decode of the CPU oracle at "
                f"{L}x{L} latents (run once), plus per step one full-size {c['num_inference_steps']}-row parental mix and "
                f"one LPIPS pair at {8 * L} px; UNet time scaled by the analytic FLOP ratio {Lf}^2 vs {L}^2 latents "
                f"(x{unet_tflop(Lf) / unet_tflop(L):.2f}), VAE/LPIPS by the pixel ratio (x{(Lf / L) ** 2:.0f}); "
                f"transition time extrapolated with the exact call counts ({c['unet_forwards'] or 198} UNet, "
                f"{c['frames'] or 15} VAE, {c.get('mixes') or 13} mixes, {c.get('lpips') or 26} LPIPS)")


def cpu_baseline_block(port, res):
    return dict(value=res["frames_per_s"], unit="frames/s", cores=port.threads, kind="port",
                sample=port.sample_text(),
                detail=dict({k: round(v, 4) for k, v in res.items() if k.startswith("t_")},
                            unet_sample_gflops=round(res["unet_sample_gflops"], 1), **port.thread_detail))


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    cfg = CONFIGS[args.config if args.config != 4 else 2]
    port = CpuPort(cfg)
    for _ in range(max(0, args.warmup)):
        port.step()
    vals = [port.step() for _ in range(max(1, args.steps))]
    fps = sum(v["frames_per_s"] for v in vals) / len(vals)
    tt = sum(v["transition_s_extrapolated"] for v in vals) / len(vals)
    last = dict(vals[-1], frames_per_s=fps)
    line = dict(metric=cfg["metric"], value=fps, unit="frames/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, ms_per_step=tt * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="f32", data="synthetic", config=workload_config(cfg, "host CPU"), impl="reference",
                cpu_baseline=cpu_baseline_block(port, last),
                e2e=dict(value=fps, unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0,
                extrapolated=True)
    print(json.dumps(line), flush=True)


def workload_config(cfg, parallelism):
    return dict(workload=cfg["workload"], frames=cfg["frames"], unet_forwards=cfg["unet_forwards"],
                cfg_batch=cfg["cfg_batch"], latent=f"{cfg['latent']}x{cfg['latent']}",
                weights=f"random-init SDXL-{cfg['model']} shape", seeds=cfg["seeds"], l2=L2_NOTE,
                parallelism=parallelism)


# ---------------------------------------------------------------------------------------------
def tree_fingerprint(be):
    """sha1 over the finished tree: fracts, injection indices and every branch's final latents (bytes)."""
    import numpy as np
    import torch
    h = hashlib.sha1()
    h.update(np.asarray(be.tree_fracts, dtype=np.float64).tobytes())
    h.update(np.asarray(be.tree_idx_injection, dtype=np.int64).tobytes())
    finals = torch.stack([t[-1].reshape(-1) for t in be.tree_latents], 0).contiguous()
    h.update(finals.cpu().numpy().tobytes())
    return h.hexdigest()


DUMP_FRAME_VALUES = 1 << 23     # 32 MB of float32 frame samples; the final latents add at most 8 MB (config 3)


def dump_outputs(out_dir, frames, be):
    """Write what the last timed step computed as .npy files under ``out_dir``:
    ``frames`` float32 [n_frames, k]: the returned uint8 RGB frames at k pixel-channel positions drawn once from a
    fixed seed (the same positions in every frame; all of them when the frames are small enough),
    ``final_latents`` float32 [n_branches, ...]: every branch's final latents in tree order,
    ``tree_fracts`` float64 [n_branches]: the branches' mixing fractions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    fr = torch.stack(frames).reshape(len(frames), -1)
    k = min(fr.shape[1], DUMP_FRAME_VALUES // len(frames))
    idx = np.sort(np.random.default_rng(0).choice(fr.shape[1], k, replace=False))
    np.save(os.path.join(out_dir, "frames.npy"), fr[:, torch.from_numpy(idx).to(fr.device)].float().cpu().numpy())
    finals = torch.stack([t[-1] for t in be.tree_latents], 0)
    np.save(os.path.join(out_dir, "final_latents.npy"), finals.float().cpu().numpy())
    np.save(os.path.join(out_dir, "tree_fracts.npy"), np.asarray(be.tree_fracts, dtype=np.float64))


def run_ours(args):
    import torch
    rank, local_rank, world = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device for --impl ours"
    torch.cuda.set_device(local_rank)
    dev = f"cuda:{local_rank}"
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))
    from latentblending_b200 import BlendingEngine, SyntheticSDXLPipe, ops
    from latentblending_b200._cabi import OP_ATTENTION, OP_GEMM, OP_GROUPNORM, OP_LAYERNORM
    cfg = CONFIGS[args.config]
    pk = peaks()
    name = "stabilityai/sdxl-turbo" if cfg["model"] == "turbo" else "stabilityai/stable-diffusion-xl-base-1.0"
    pipe = SyntheticSDXLPipe(name, dev, seed=0)
    be = BlendingEngine(pipe)
    if cfg["model"] == "turbo":
        # ancestral noise per (seeds, branch position, step) instead of global-RNG draws: the tree then does not depend on
        # the order branches are computed in (lockstep speculation, sharding), so fingerprints compare across --gpus
        be.deterministic_noise = True
    be.set_negative_prompt(NEG)
    be.set_prompt1(PROMPTS[0])
    be.set_prompt2(PROMPTS[1])
    if cfg["branch1_crossfeed"]:
        be.set_branch1_crossfeed(*cfg["branch1_crossfeed"])
    if args.config == 4:
        be.set_branching(t_compute_max_allowed=args.t_compute)
    elif cfg["model"] == "turbo":
        be.set_branching(nmb_max_branches=cfg["nmb_max_branches"])
    else:
        be.set_branching(depth_strength=cfg["depth_strength"], nmb_max_branches=cfg["nmb_max_branches"])
    if cfg["stems"] is not None:
        assert [int(v) for v in be.list_nmb_stems] == cfg["stems"], be.list_nmb_stems

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 0
        for _ in range(steps):
            n += fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms / 1e3, n

    step_frames = []        # the frames returned in the latest step

    def one_job(api):
        """One bench step.  Configs 2/3/5: one transition.  Config 4: the 8-prompt loop (7 transitions)."""
        be.output_device_frames = not api
        step_frames.clear()
        if args.config != 4:
            if api:
                be.set_prompt1(PROMPTS[0])
                be.set_prompt2(PROMPTS[1])
            step_frames.extend(be.run_transition(fixed_seeds=list(cfg["seeds"])))
            return len(step_frames)
        for i in range(len(PROMPTS_MULTI) - 1):
            if i == 0:
                be.set_prompt1(PROMPTS_MULTI[0])
                be.set_prompt2(PROMPTS_MULTI[1])
            else:
                be.swap_forward()
                be.set_prompt2(PROMPTS_MULTI[i + 1])
            step_frames.extend(be.run_transition(recycle_img1=i > 0, fixed_seeds=[420 + i, 421 + i]))
        return len(step_frames)

    for _ in range(max(args.warmup, 0)):
        one_job(False)
    sampler = ClockSampler(local_rank)
    sampler.start()
    try:
        ops.LAUNCHES[0] = 0
        sec, frames = timed(lambda: one_job(False), args.steps)
        launches = ops.LAUNCHES[0]
    finally:
        clocks = sampler.stop()
    fps = frames / sec
    fingerprint = tree_fingerprint(be)          # of the last timed transition (identical every step: fixed seeds)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_frames, be)
    stems_run = [int(v) for v in be.list_nmb_stems]
    # e2e through the public API with host buffers
    one_job(True)
    pipe.h2d_bytes = 0
    be.d2h_bytes = 0
    sec_e, frames_e = timed(lambda: one_job(True), args.steps)
    e2e = dict(value=frames_e / sec_e, unit="frames/s", h2d_bytes_per_step=pipe.h2d_bytes // max(1, args.steps),
               d2h_bytes_per_step=be.d2h_bytes // max(1, args.steps))

    # roofline of the dominant kernel (gemm_tc_kernel): all GEMM launches of one UNet forward, replayed
    # back to back on the launching stream between CUDA events
    Bp, Lp = cfg["cfg_batch"], cfg["latent"]
    plan = be.dh.unet.plan(Bp, Lp, Lp)
    work = plan.prog_step.work()
    breakdown = {}
    for name_, kinds in (("gemm", [OP_GEMM]), ("attention", [OP_ATTENTION]), ("norms", [OP_GROUPNORM, OP_LAYERNORM]),
                         ("all", list(range(1, 11)))):
        for _ in range(2):
            plan.prog_step.run_kinds(kinds, 500.0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps):
            n_l = plan.prog_step.run_kinds(kinds, 500.0)
        e1.record()
        torch.cuda.synchronize()
        breakdown[name_] = dict(ms=e0.elapsed_time(e1) / reps, launches=n_l)
    # K1 (crossfeed / parental mix) in its batched form: 2048 rows x 65536 fp16 (805 MB through the kernel, > L2)
    mp0 = torch.randn(2048, 4 * 128 * 128, device=dev).half()
    mp1 = torch.randn(2048, 4 * 128 * 128, device=dev).half()
    mout = torch.empty_like(mp0)
    for _ in range(3):
        ops.slerp_rows(mp0, mp1, 0.4, out=mout)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        ops.slerp_rows(mp0, mp1, 0.4, out=mout)
    e1.record()
    torch.cuda.synchronize()
    mix_s = e0.elapsed_time(e1) / 10 * 1e-3
    mix_gbs = mp0.numel() * 6 / mix_s / 1e9
    del mp0, mp1, mout
    gemm_tf = work["gemm_flops"] / (breakdown["gemm"]["ms"] * 1e-3) / 1e12
    attn_tf = work["attn_flops"] / (breakdown["attention"]["ms"] * 1e-3) / 1e12
    norm_gbs = work["norm_bytes"] / max(breakdown["norms"]["ms"] * 1e-3, 1e-9) / 1e9
    peak_tf, peak_burst = pk["bf16_tflops_sustained"], pk["bf16_tflops"]
    tr = measured_traffic()
    roofline = dict(kernel="gemm_tc_kernel (tcgen05 GEMM / implicit-GEMM conv)", bound="tensor", achieved=gemm_tf,
                    peak=peak_tf, unit="TFLOP/s", frac=gemm_tf / peak_tf, frac_of_burst_peak=gemm_tf / peak_burst,
                    traffic=tr.get("gemm", {}).get("dram_bytes_per_launch"),
                    traffic_source=tr.get("gemm", {}).get("source"),
                    algorithmic_bytes_per_launch=work["gemm_bytes"] / max(1, breakdown["gemm"]["launches"]),
                    peak_source=f"{pk['source']} bf16_tflops_sustained (the replay follows minutes of load under the "
                                f"power cap; burst peak {peak_burst} also given)",
                    algorithmic_flops_per_unet_forward=work["gemm_flops"],
                    avg_launch_us=breakdown["gemm"]["ms"] * 1e3 / max(1, breakdown["gemm"]["launches"]),
                    launches_per_unet_forward=breakdown["gemm"]["launches"],
                    unet_forward_breakdown_ms={k: round(v["ms"], 3) for k, v in breakdown.items()},
                    unet_forward_launches={k: v["launches"] for k, v in breakdown.items()},
                    attention=dict(kernel="attn_tc_kernel (tcgen05 QK^T / PV, head dim 64)", achieved=attn_tf,
                                   frac=attn_tf / peak_tf, flops=work["attn_flops"],
                                   note="all attention launches of one UNet forward incl. cross-attention (77 keys)"),
                    norms=dict(kernel="gn_stats/gn_apply/ln kernels", bound="hbm", achieved=norm_gbs,
                               peak=pk["hbm_gbs"], unit="GB/s", frac=norm_gbs / pk["hbm_gbs"],
                               algorithmic_bytes=work["norm_bytes"]),
                    mix=dict(kernel="slerp_l2_kernel (K1 parental / crossfeed mix, batched 2048 x 65536 fp16)",
                             bound="hbm", achieved=mix_gbs, peak=pk["hbm_gbs"], unit="GB/s", frac=mix_gbs / pk["hbm_gbs"],
                             algorithmic_bytes_per_element=6, launch_us=mix_s * 1e6,
                             traffic=tr.get("mix", {}).get("dram_bytes_per_launch"),
                             traffic_source=tr.get("mix", {}).get("source")))

    par = "single GPU" if world == 1 else (f"branch-sharded x{world}: one speculative candidate per rank, CFG halves "
                                           f"split over GPU pairs for the outer trajectories (>= 4 ranks) and the last stems of a level")
    wc = workload_config(cfg, par)
    wc["stems"] = stems_run
    wc["speculative_batch"] = be._speculation_width() if world == 1 else 1
    if getattr(be, "spec_stats", None) and world == 1:
        wc["speculation"] = dict(be.spec_stats, lifetime_second_candidates_used_of_computed=list(be._spec_hits))
    if args.config == 4:
        wc.update(frames=frames // max(1, args.steps), t_compute_max_allowed=args.t_compute,
                  dt_unet_step=round(float(be.dt_unet_step), 5), dt_vae=round(float(be.dt_vae), 5))
    line = dict(metric=cfg["metric"], value=fps, unit="frames/s", n_gpus=world, steps=args.steps, warmup=args.warmup,
                ms_per_step=sec / max(1, args.steps) * 1e3, higher_is_better=True, scaling="strong",
                vs_baseline=None, dtype="f16", data="synthetic", config=wc, clocks=clocks, e2e=e2e,
                gpu_launches=launches, roofline=roofline, impl="ours", fingerprint=fingerprint,
                shard_stats=getattr(be, "shard_stats", None))
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            port = CpuPort(cfg if args.config != 4 else CONFIGS[2])
            line["cpu_baseline"] = cpu_baseline_block(port, port.step())
        except Exception as ex:   # the baseline is a reported number, never a reason to lose the bench line
            line["cpu_baseline"] = dict(value=None, unit="frames/s", cores=host_cpu_budget(), kind="port",
                                        sample=f"failed: {ex!r}")
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--t-compute", type=float, default=6.0,
                    help="config 4: t_compute_max_allowed per transition (the reference default is 20 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/*.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
