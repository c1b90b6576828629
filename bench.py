"""bench.py — headline benchmark of the CFG++ sampling hot path (driver contract in the task statement).

    python bench.py --gpus N --steps K --warmup W            # ours: hand-written sm_100a path behind the C ABI
    python bench.py --impl reference --gpus N --steps K ...  # reference arm: the repo's CPU eager path (oracle)
    python bench.py --config {sdxl_b2,sd15_b4,sdxl_dpmpp_64,lightning_b8}   # the other BASELINE.json configs
    python bench.py ... --dump-outputs DIR   # also save the last timed trajectory's result as DIR/latents.npy (fp32)

Default workload = BASELINE.json's metric config (configs[2]): images/sec, device-timed, SDXL 1024x1024 NFE=50
ddim_cfg++ lambda=0.6, batch 2 per GPU. N>1 shards independent prompts over ranks (weak scaling, no per-step
collective, one NCCL broadcast of the UNet weights at init). One "step" = one full sampling trajectory of one batch
(NFE fused UNet+CFG++ steps): from zT resident in HBM to the final latent — text encoding and VAE decode stay on the
reference path and are outside the metric (SURVEY.md §8d).

Order of work (so that a lost run loses as little as possible): device-timed leg -> e2e leg -> roofline -> the line
so far goes to STDERR -> GPU eager baseline -> bounded CPU baseline -> the ONE JSON line on stdout. Nothing is written
under the source tree.

Inputs are seeded (weights from seed 1234, each trajectory's prompt embeddings and zT from its index), so two runs
with the same arguments see identical inputs and their --dump-outputs files can be compared across builds.

Synthetic data: no checkpoint / tokenizer exists offline, so weights are seeded synthetic under the diffusers key
names (random-init of the real architectures: SDXL 2,567,463,684 params, SD v1.5 859,520,964) and the conditioning
tensors are seeded random embeddings of the real shapes.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402
import torch  # noqa: E402

# ----------------------------------------------------------------------------------------------------------------
# workloads = BASELINE.json configs[1..4] (configs[0] is the CPU plumbing case = the cpu_baseline leg)
# ----------------------------------------------------------------------------------------------------------------
WORKLOADS = {
    "sdxl_b2": dict(family="sdxl", method="ddim_cfg++", nfe=50, lam=0.6, batch=2, latent=128,
                    metric="images/sec (device-timed) SDXL 1024x1024 NFE=50 ddim_cfg++",
                    workload="SDXL 1024x1024 ddim_cfg++ lambda=0.6 NFE=50 batch=2 per GPU (configs[2])"),
    "sd15_b4": dict(family="sd15", method="ddim_cfg++", nfe=50, lam=0.6, batch=4, latent=64,
                    metric="images/sec (device-timed) SDv1.5 512x512 NFE=50 ddim_cfg++",
                    workload="SDv1.5 512x512 ddim_cfg++ lambda=0.6 NFE=50 batch=4 per GPU (configs[1])"),
    "sdxl_dpmpp_64": dict(family="sdxl", method="dpm++_2m_cfgpp", nfe=25, lam=0.6, batch=8, latent=128,
                          metric="images/sec (device-timed) SDXL 1024x1024 NFE=25 dpm++_2m_cfgpp",
                          workload="SDXL 1024x1024 dpm++_2m_cfgpp lambda=0.6 NFE=25 (24 steps), 8 prompts per GPU "
                                   "per trajectory = prompt-batch 64 over 8 GPUs (configs[3])"),
    "lightning_b8": dict(family="sdxl_lightning", method="ddim_cfg++_lightning", nfe=4, lam=1.0, batch=8, latent=128,
                         metric="images/sec (device-timed) SDXL-Lightning 1024x1024 NFE=4 ddim_cfg++_lightning",
                         workload="SDXL-Lightning 1024x1024 ddim_cfg++_lightning lambda=1.0 NFE=4 batch=8 per GPU "
                                  "(configs[4])"),
}
DEFAULT_WORKLOAD = "sdxl_b2"
ROOFLINE_TRAFFIC_FILE = ROOT / "profiles" / "roofline_traffic.json"  # written by tools/summarize_profiles.py from ncu


def log(msg):
    print(f"[bench] {msg}", file=sys.stderr, flush=True)


# stdout carries exactly ONE line — the JSON record. Libraries write there too (NCCL prints its version banner on fd 1
# from C), so fd 1 is pointed at stderr for the whole run and the record goes to a saved copy of the real stdout.
_REAL_STDOUT = None


def _capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"tflops": d.get("bf16_tflops_sustained", 1445.3), "hbm": d.get("hbm_gbs", 6587.7), "source": "measured"}
    return {"tflops": 1400.0, "hbm": 6650.0, "source": "fallback"}


def unet_config(family):
    from cfgpp_b200 import config as C
    return C.sd15_config() if family == "sd15" else C.sdxl_config()


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": statistics.median(pw) if pw else None, "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------------------------
# synthetic workload
# ----------------------------------------------------------------------------------------------------------------
def synthetic_conditioning(cfg, wl, seed, pin=True):
    """Host-side (pinned) conditioning + zT for one batch, shapes of latent_sdxl.py:222-257 / :289. With
    cfg_guidance in {0, 1} (Lightning) the reference passes the added conditions un-duplicated (:249-252)."""
    batch, latent = wl["batch"], wl["latent"]
    g = torch.Generator(device="cpu").manual_seed(seed)
    t = {"uc": torch.randn(batch, 77, cfg.cross_attention_dim, generator=g).half(),
         "c": torch.randn(batch, 77, cfg.cross_attention_dim, generator=g).half()}
    if cfg.addition_embed_type == "text_time":
        rows = batch if wl["lam"] in (0.0, 1.0) else 2 * batch
        t["pooled"] = torch.randn(rows, cfg.pooled_dim, generator=g).half()
        t["time_ids"] = torch.tensor([[1024., 1024., 0., 0., 1024., 1024.]] * rows).half()
    g2 = torch.Generator(device="cpu").manual_seed(42 + seed)
    t["zT"] = torch.randn(batch, 4, latent, latent, generator=g2)
    if pin and torch.cuda.is_available():
        t = {k: v.pin_memory() for k, v in t.items()}
    return t


def nbytes(*ts):
    return int(sum(x.numel() * x.element_size() for x in ts))


def make_solver(wl, cfg, dev, sd):
    ns = argparse.Namespace(num_sampling=wl["nfe"])
    if wl["family"] == "sd15":
        from cfgpp_b200.latent_diffusion import get_solver
        return get_solver(wl["method"], solver_config=ns, device=dev, model_key="synthetic:1234", state_dict=sd)
    from cfgpp_b200.latent_sdxl import get_solver
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # Lightning: "checkpoint not found; using seeded synthetic weights"
        return get_solver(wl["method"], solver_config=ns, device=dev, state_dict=sd,
                          **({} if wl["family"] == "sdxl_lightning" else {"model_key": "synthetic:1234"}))


def solve(solver, wl, t):
    """One trajectory through the reference-facing solver API (reverse_process of the registered --method)."""
    side = 8 * wl["latent"]
    if wl["family"] == "sd15":
        return solver.reverse_process(t["uc"], t["c"], wl["lam"], t["zT"])
    add = {"text_embeds": t["pooled"], "time_ids": t["time_ids"]}
    return solver.reverse_process(t["uc"], t["c"], wl["lam"], add, (side, side), zT=t["zT"])


# ----------------------------------------------------------------------------------------------------------------
# CPU baseline = the oracle ("repo's own CPU eager path"), bounded sample
# ----------------------------------------------------------------------------------------------------------------
def _host_ram_gb():
    try:
        import psutil
        avail = psutil.virtual_memory().available / 2**30
    except Exception:  # noqa: BLE001
        avail = 64.0
    try:
        lim = Path("/sys/fs/cgroup/memory.max").read_text().strip()
        if lim.isdigit():
            avail = min(avail, int(lim) / 2**30)
    except Exception:  # noqa: BLE001
        pass
    return avail


def pick_threads():
    """Thread count for the CPU leg: the affinity mask can be far larger than the CPU time the container really gets
    (round 1: 128 visible cores ran a GEMM at 160 GFLOP/s), and oversubscribed threads make the oracle slower, so a
    short fp32 GEMM probe picks the fastest of {all, 64, 32, 16, 8} threads. Returns (threads, probe GFLOP/s)."""
    avail = len(os.sched_getaffinity(0))
    a, b = torch.randn(2048, 5120), torch.randn(5120, 1280)
    best = (avail, 0.0)
    for nt in sorted({n for n in (avail, 64, 32, 16, 8) if n <= avail}, reverse=True):
        torch.set_num_threads(nt)
        torch.mm(a, b)
        t0 = time.perf_counter()
        for _ in range(2):
            torch.mm(a, b)
        gf = 2 * 2 * 2048 * 5120 * 1280 / (time.perf_counter() - t0) / 1e9
        if gf > best[1] * 1.1:   # prefer more threads unless fewer are clearly faster
            best = (nt, gf)
    torch.set_num_threads(best[0])
    return best


class CpuOracle:
    """fp32 oracle UNet on the host cores (the reference's `pipe_dtype=torch.float32` CPU path). Built ONCE, straight
    in fp32 on the CPU with a cheap deterministic fill (timing does not depend on the weight values; no state dict and
    no second copy are ever held: SDXL = 10.3 GB, SD v1.5 = 3.4 GB of host RAM). Sample = one UNet sample-forward at a
    reduced latent, scaled to the workload's latent by algorithmic FLOPs."""

    def __init__(self, family):
        import dataclasses
        from oracle import unet as O
        self.cores, self.probe_gflops = pick_threads()
        if family != "sd15" and _host_ram_gb() < 20.0:
            log("host RAM < 20 GB: CPU sample falls back to the SD v1.5 UNet")
            family = "sd15"
        self.family = family
        self.cfg = unet_config(family)
        ocfg = O.UNetConfig(**{f.name: getattr(self.cfg, f.name) for f in dataclasses.fields(O.UNetConfig)})
        t0 = time.perf_counter()
        with torch.device("meta"):
            m = O.UNet2DConditionModel(ocfg)
        m = m.to_empty(device="cpu")
        with torch.no_grad():
            for i, p in enumerate(m.parameters()):
                p.fill_(0.02 if p.dim() > 1 else (1.0 if i % 2 == 0 else 0.0))
        self.m = m.eval().requires_grad_(False)
        self.build_s = time.perf_counter() - t0
        # algorithmic FLOPs per sample-forward (SURVEY §8d) at the full latent, and their self-attention part
        self.f_full, self.f_attn, self.full_latent = ((0.8032, 0.1225, 64) if family == "sd15"
                                                      else (6.7612, 0.7516, 128))

    def sample(self, latent):
        """seconds of ONE sample-forward at the FULL latent, measured at `latent` and FLOP-scaled."""
        cfg = self.cfg
        g = torch.Generator().manual_seed(0)
        x = torch.randn(1, 4, latent, latent, generator=g)
        ctx = torch.randn(1, 77, cfg.cross_attention_dim, generator=g)
        add = None
        if cfg.addition_embed_type == "text_time":
            add = {"text_embeds": torch.randn(1, cfg.pooled_dim, generator=g),
                   "time_ids": torch.tensor([[1024., 1024., 0., 0., 1024., 1024.]])}
        with torch.no_grad():
            t0 = time.perf_counter()
            self.m(x, torch.tensor(501), ctx, add)
            dt = time.perf_counter() - t0
        r = self.full_latent // latent  # convs / token GEMMs shrink r^2, self-attention r^4
        f_small = (self.f_full - self.f_attn) / r ** 2 + self.f_attn / r ** 4
        return dt * self.f_full / f_small, dt


def cpu_baseline(wl, max_samples=1):
    """images/sec of the reference's CPU eager path for workload `wl`: one image = NFE' x 2 sample-forwards."""
    fam = "sd15" if wl["family"] == "sd15" else "sdxl"
    orc = CpuOracle(fam)
    # full-size latent when the GEMM probe says one forward fits ~45 s; otherwise the half-size latent, FLOP-scaled
    # (small latents run less efficiently, so the scaled figure, if anything, UNDER-states the CPU path's speed)
    est_full = orc.f_full * 1e3 / max(0.5 * orc.probe_gflops, 1e-3)
    latent = orc.full_latent if est_full <= 45.0 else orc.full_latent // 2
    best, raw = None, None
    for _ in range(max_samples):
        t_full, dt = orc.sample(latent)
        if best is None or t_full < best:
            best, raw = t_full, dt
    steps = wl["nfe"] - 1 if wl["method"].startswith("dpm++") else wl["nfe"]
    scale = 1.0
    if orc.family != fam:  # RAM fallback: SD v1.5 module timed, scaled to SDXL by algorithmic FLOPs
        scale = 6.7612 / 0.8032
    value = 1.0 / (2 * steps * best * scale)
    how = (f"1 {orc.family.upper()} UNet sample-forward (batch 1, fp32, {orc.cores} threads) at {latent}x{latent} latent "
           f"= {raw:.1f} s" + (f", scaled to {orc.full_latent}x{orc.full_latent} by algorithmic FLOPs = {best:.1f} s"
                               if latent != orc.full_latent else "") +
           f"; one image = {2 * steps} such forwards" + ("; SD v1.5 module scaled to SDXL FLOPs (host RAM)" if scale != 1 else ""))
    res = {"value": value, "unit": "images/sec", "cores": orc.cores, "cores_visible": len(os.sched_getaffinity(0)),
           "kind": "port", "sample": how, "seconds_per_unet_forward": best * scale, "sample_seconds": raw,
           "probe_gflops": orc.probe_gflops}
    del orc
    return res


# ----------------------------------------------------------------------------------------------------------------
def run_reference_arm(args, wl):
    """--impl reference: the reference's own CPU implementation of the path = the oracle port (the reference itself
    cannot be imported: diffusers is absent and not installable offline), all host threads, bounded samples."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_baseline(wl, max_samples=max(1, min(args.steps, 2)))
    line = {"impl": "reference", "metric": wl["metric"], "value": r["value"], "unit": "images/sec", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wl["batch"] / r["value"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["workload"], "global_batch": wl["batch"] * args.gpus,
                       "parallelism": f"dp{args.gpus}"},
            "cpu_baseline": r,
            "e2e": {"value": r["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ----------------------------------------------------------------------------------------------------------------
def run_ours(args, wl):
    import torch.distributed as dist
    from cfgpp_b200 import weights as Wt
    from cfgpp_b200 import dist as D
    from cfgpp_b200.engine import NativeUNet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (ours) needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = unet_config(wl["family"])
    NFE, BATCH, LATENT = wl["nfe"], wl["batch"], wl["latent"]
    nsteps = NFE - 1 if wl["method"].startswith("dpm++") else NFE
    # ---- weights: rank 0 generates, ONE bucketed NCCL broadcast at init makes replicas bit-identical -------------
    sd = Wt.synthetic_state_dict(cfg, seed=1234, device=dev) if rank == 0 else None
    if world > 1:
        sd = D.broadcast_state_dict(sd, Wt.unet_param_specs(cfg), dev, src=0)
    solver = make_solver(wl, cfg, dev, sd)
    eng: NativeUNet = solver.unet
    eng.prepare(BATCH, LATENT, LATENT)
    stats = eng.plan_stats

    # every trajectory uses its own prompt / zT (rank r owns items r, r+W, ...: D.shard_indices)
    n_traj = args.warmup + args.steps
    items = D.shard_indices(world * n_traj, rank, world)
    host = [synthetic_conditioning(cfg, wl, seed=it) for it in items]
    dev_in = [{k: v.to(dev) for k, v in h.items()} for h in host]
    torch.cuda.synchronize()

    def trajectory_device(i):
        """inputs already resident in HBM (the `value` leg); the result stays on the device."""
        return solve(solver, wl, dev_in[i])

    def trajectory_e2e(i):
        """public solver API with HOST buffers: H2D of this step's inputs, D2H of the result (the `e2e` leg)."""
        t = {k: v.to(dev, non_blocking=True) for k, v in host[i].items()}
        return solve(solver, wl, t).cpu()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, first, count):
        """(ms over `count` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(first, first + count):
            out = fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), out

    for i in range(args.warmup):
        trajectory_device(i)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_dev, last = timed(trajectory_device, args.warmup, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        # the final latents of the last timed trajectory, [batch, 4, latent, latent] (<= 2 MB for every workload)
        args.dump_outputs.mkdir(parents=True, exist_ok=True)
        name = "latents" if world == 1 else f"latents_rank{rank}"
        np.save(args.dump_outputs / f"{name}.npy", last.float().cpu().numpy())
    del last
    # e2e leg (reuses the same warm engine; its own warm-up trajectory first)
    trajectory_e2e(0)
    ms_e2e, _ = timed(trajectory_e2e, args.warmup, args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    imgs = BATCH * args.steps * world
    value = imgs / (ms_dev / 1e3)
    e2e_val = imgs / (ms_e2e / 1e3)
    peaks = measured_peaks()
    log(f"value {value:.4f} img/s, e2e {e2e_val:.4f} img/s")

    # ---- roofline of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv), measured live with CUDA events ----
    d = dev_in[0]
    if "pooled" in d:
        eng.set_prompt(torch.cat([d["uc"], d["c"]]), d["pooled"], d["time_ids"].float())
    else:
        eng.set_prompt(torch.cat([d["uc"], d["c"]]))
    eng.profile_forward(d["zT"], 501.0)
    prof = eng.profile_forward(d["zT"], 501.0)
    by_kind = {0: [0.0, 0.0, 0], 1: [0.0, 0.0, 0], 2: [0.0, 0.0, 0], 3: [0.0, 0.0, 0]}
    for _, kind, fl, ms in prof:
        by_kind[kind][0] += fl
        by_kind[kind][1] += ms
        by_kind[kind][2] += 1
    gemm_fl = by_kind[0][0] + by_kind[1][0]
    gemm_ms = by_kind[0][1] + by_kind[1][1]
    gemm_n = by_kind[0][2] + by_kind[1][2]
    tot_ms = sum(v[1] for v in by_kind.values())
    achieved = gemm_fl / (gemm_ms / 1e3) / 1e12
    traffic, traffic_src = None, "no ncu --set full capture of this workload is committed"
    if ROOFLINE_TRAFFIC_FILE.exists():
        tj = json.loads(ROOFLINE_TRAFFIC_FILE.read_text()).get(args.config)
        if tj:
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
    roofline = {"bound": "tensor", "kernel": "gemm_kernel<BN,GEGLU,CL> (tcgen05 GEMM + implicit-GEMM conv3x3)",
                "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": achieved / peaks["tflops"],
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peaks["source"] + " (bf16 sustained)",
                "flops_per_launch": gemm_fl / max(gemm_n, 1), "launches_per_forward": gemm_n,
                "avg_launch_us": 1e3 * gemm_ms / max(gemm_n, 1), "share_of_step": gemm_ms / tot_ms,
                "by_kind_ms": {"linear_gemm": by_kind[0][1], "conv3x3": by_kind[1][1], "attention": by_kind[2][1],
                               "norm_elementwise": by_kind[3][1]},
                "by_kind_tflops": {"linear_gemm": by_kind[0][0] / max(by_kind[0][1], 1e-9) / 1e9,
                                   "conv3x3": by_kind[1][0] / max(by_kind[1][1], 1e-9) / 1e9,
                                   "attention": by_kind[2][0] / max(by_kind[2][1], 1e-9) / 1e9}}
    # executed FLOPs: `step_flops` every step + `prompt_flops` once per trajectory; the reference-equivalent
    # algorithmic figure charges the K/V projections to every step (diffusers recomputes them)
    per_traj_exec = stats["step_flops"] * nsteps + stats["prompt_flops"]
    per_traj_algo = eng.forward_flops * nsteps
    sec = ms_dev / 1e3 / args.steps
    launches = int((eng.launches_per_step * nsteps + stats["prompt_launches"]) * args.steps)

    line = {"metric": wl["metric"], "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": wl["workload"], "name": args.config,
                       "global_batch": BATCH * world, "parallelism": f"dp{world} (independent prompts, no per-step collective)",
                       "step": f"one full trajectory of one batch ({nsteps} fused UNet uncond+cond + CFG++/scheduler steps)",
                       "l2": "inputs larger than L2 (fp16 weights streamed every UNet forward: 5.1 GB SDXL / 1.7 GB SD v1.5; 126 MB L2)"},
            "e2e": {"value": e2e_val, "unit": "images/sec",
                    "h2d_bytes_per_step": nbytes(*host[0].values()),
                    "d2h_bytes_per_step": BATCH * 4 * LATENT * LATENT * (2 if wl["method"].startswith("dpm++") else 4),
                    "api": f"get_solver('{wl['method']}').reverse_process(...) with pinned host inputs, result .cpu()"},
            "gpu_launches": launches,
            "clocks": clocks, "roofline": roofline,
            "unet_tflops_per_gpu": {"executed": per_traj_exec / sec / 1e12, "algorithmic": per_traj_algo / sec / 1e12},
            "unet_frac_of_peak": per_traj_exec / sec / 1e12 / peaks["tflops"],
            "forward_tflop": {"executed_per_step": stats["step_flops"] / 1e12,
                              "once_per_prompt": stats["prompt_flops"] / 1e12,
                              "algorithmic_per_step": eng.forward_flops / 1e12}}

    # ---- VAE decode of one batch of final latents (outside the metric; the step after the path, SURVEY §8 f2) --------
    try:
        dec = getattr(getattr(solver, "vae", None), "decoder", None)
        if dec is not None:
            zfin = trajectory_device(args.warmup)
            dec.decode_fp16(zfin)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                dec.decode_fp16(zfin)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 3
            st = dec.stats
            line["vae_decode"] = {"ms_per_batch": ms, "images": BATCH, "tflops": st["flops"] / (ms / 1e3) / 1e12,
                                  "share_of_trajectory": ms / (ms_dev / args.steps),
                                  "what": "native AutoencoderKL decoder (cfgpp_vae_decode), device-timed, not part of `value`"}
            del dec, zfin
    except Exception as e:  # noqa: BLE001 — never lose the measured line to an optional leg
        line["vae_decode"] = {"error": repr(e)[:200]}

    # ---- prompt conditioning of one batch (outside the metric; the step before the path, SURVEY §8 f3) -----------------
    try:
        from cfgpp_b200.text_encoder import ClipConditioner
        towers = [t for t in (getattr(solver, "text_enc_1", None), getattr(solver, "text_enc_2", None),
                              getattr(solver, "text_encoder", None)) if isinstance(t, ClipConditioner)]
        if towers:
            prompts = [""] + [f"a photo of an astronaut riding horse number {i} on mars" for i in range(BATCH)]

            def encode_all():
                return [t.encode_batch(prompts) for t in towers]
            encode_all()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                encode_all()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 3
            fl = sum(t.encoder.stats["flops"] for t in towers)
            line["text_encode"] = {"ms_per_batch": ms, "prompts": len(prompts), "towers": [t.encoder.cfg.name for t in towers],
                                   "tflops": fl / (ms / 1e3) / 1e12, "share_of_trajectory": ms / (ms_dev / args.steps),
                                   "what": "native CLIP text towers (cfgpp_clip_encode) incl. host tokenisation, "
                                           "device-timed, not part of `value`"}
    except Exception as e:  # noqa: BLE001
        line["text_encode"] = {"error": repr(e)[:200]}

    def checkpoint_line():
        print("[bench partial] " + json.dumps(line), file=sys.stderr, flush=True)

    checkpoint_line()
    # ---- baselines measured beside it (rank 0, N=1 only) ---------------------------------------------------------
    if world == 1 and not args.no_baselines:
        from cfgpp_b200.latent_sdxl import release_engines
        del solver, eng
        release_engines()
        torch.cuda.empty_cache()
        try:
            line["gpu_eager_baseline"] = gpu_eager_baseline(cfg, wl, sd, dev)
            line["speedup_vs_gpu_eager"] = value / line["gpu_eager_baseline"]["value"]
        except Exception as e:  # noqa: BLE001 — a failing baseline must not cost the measured line
            line["gpu_eager_baseline"] = {"error": repr(e)[:200]}
        del sd
        torch.cuda.empty_cache()
        checkpoint_line()
        try:
            line["cpu_baseline"] = cpu_baseline(wl)
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": repr(e)[:200], "value": None, "unit": "images/sec",
                                    "cores": len(os.sched_getaffinity(0)), "kind": "port", "sample": "failed"}
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def gpu_eager_baseline(cfg, wl, sd, dev, n_time=6, n_warm=2):
    """The north-star comparator ("reference CUDA path" stand-in, BASELINE.md §3): the restated diffusers op sequence
    + the reference-style Python step loop (incl. its per-step host syncs) under torch.autocast('cuda', fp16) on the
    same GPU and inputs. Times `n_time` steps after `n_warm` and scales to the trajectory (every step costs the same)."""
    import dataclasses
    from oracle import samplers as OSm, schedule as OS, unet as O
    ocfg = O.UNetConfig(**{f.name: getattr(cfg, f.name) for f in dataclasses.fields(O.UNetConfig)})
    m = O.build_unet(ocfg, sd, dtype=torch.float16, device=dev)
    h = synthetic_conditioning(cfg, wl, seed=0, pin=False)
    uc, c, zT = h["uc"].to(dev), h["c"].to(dev), h["zT"].to(dev)
    add = {"text_embeds": h["pooled"].to(dev), "time_ids": h["time_ids"].to(dev)} if "pooled" in h else None
    if add is not None and add["text_embeds"].shape[0] == wl["batch"] and wl["batch"] > 1:
        # un-duplicated added conditions (cfg_guidance == 1) only broadcast for ONE image in diffusers: duplicate
        add = {k: torch.cat([v, v]) for k, v in add.items()}
    kind = "lightning" if wl["family"] == "sdxl_lightning" else "ddim"
    n_time = min(n_time, wl["nfe"] - n_warm) if wl["nfe"] > n_warm + 1 else 1
    n_warm = min(n_warm, max(1, wl["nfe"] - n_time))

    def run(nsteps):
        tb = OS.make_tables(wl["nfe"], kind)
        extra = 1 if wl["method"].startswith("dpm++") else 0   # the DPM++ loop runs len(timesteps) - 1 steps
        tb = dataclasses.replace(tb, timesteps=tb.timesteps[:nsteps + extra])
        with torch.autocast("cuda", dtype=torch.float16):
            if wl["family"] == "sd15":
                return OSm.sd15_ddim_cfgpp(m, tb, zT, uc, c, wl["lam"])
            if wl["method"].startswith("dpm++"):
                return OSm.sdxl_dpmpp_2m_cfgpp(m, tb, zT, uc, c, wl["lam"], add)
            if wl["family"] == "sdxl_lightning":
                return OSm.sdxl_ddim_cfgpp_lightning(m, tb, zT, uc, c, wl["lam"], add)
            return OSm.sdxl_ddim_cfgpp(m, tb, zT, uc, c, wl["lam"], add)

    run(n_warm)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    run(n_time)
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / n_time
    nsteps = wl["nfe"] - 1 if wl["method"].startswith("dpm++") else wl["nfe"]
    return {"value": wl["batch"] / (nsteps * ms_step / 1e3), "unit": "images/sec", "ms_per_unet_step": ms_step,
            "what": "restated diffusers UNet + reference step loop, torch eager, autocast fp16, same GPU"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=str, default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--no-baselines", action="store_true", help="skip the GPU-eager and CPU baselines at N=1")
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="write the last timed trajectory's final latents to DIR/latents.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours (the reference arm times single UNet forwards, not trajectories)")
    _capture_stdout()
    wl = WORKLOADS[args.config]
    if args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
