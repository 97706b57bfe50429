#!/usr/bin/env python
"""Benchmark of the MLD sampling path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--config headline|1prompt|action512|novae1024] [--scaling weak|strong] [--dump-outputs DIR]

Default (`--config headline`, the driver's line): motions/sec @ 50-step DDIM text-to-motion, batch 256
(BASELINE.json configs[2]: 77-token CLIP context, latent 1x256, decode to 196x263, joints).  One "step" = one
full pass of the hot path over one batch of synthetic input: 50 x (denoiser on 2B sequences + CFG + DDIM
update) + VAE decode + feats2joints (+ the all-gather of finished motions when N > 1, through the C ABI:
mldb_sample_gather).  Rank 0 prints ONE JSON line.  The other BASELINE configs (`--config`) print the same line
for their own workload; `--scaling strong` shards a fixed total batch instead of B per GPU.
``--impl reference`` times the CPU restatement of the reference path (the oracle, pinned against the
reference's own modules; the reference itself is Python and does not exist on the GPU box) on a bounded sample
of the same workload.
``--dump-outputs DIR`` writes what the timed path returned in its last step as ``DIR/<name>.npy`` (float32), so
that two builds can be compared output for output on the same seeded inputs.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree, which may be read-only

_T0 = time.time()


def _log(msg: str):
    print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------ workloads
# FLOP per motion = algorithmic model math as the reference executes it (SURVEY.md section 8d).
WORKLOADS = {
    "headline": dict(
        metric="motions/sec @ 50-step DDIM text-to-motion, batch 256", B=256, S=77, T=196, steps=50, total_fixed=False,
        flop_per_motion=132.77e9, cpu_sample=32,
        workload="text-to-motion B=256/GPU, 77-token CLIP ctx, 50 DDIM steps (CFG 7.5), decode 196x263, joints"),
    "1prompt": dict(
        metric="motions/sec @ 50-step DDIM text-to-motion, single prompt", B=1, S=77, T=196, steps=50, total_fixed=False,
        flop_per_motion=132.77e9, cpu_sample=1,
        workload="text-to-motion single prompt (B=1), 77-token CLIP ctx, 50 DDIM steps (CFG 7.5), decode 196x263, joints"),
    "action512": dict(
        metric="motions/sec @ 50-step DDIM action-to-motion, batch 512", B=512, S=1, T=60, steps=50, total_fixed=True,
        flop_per_motion=8.36e9, cpu_sample=64,
        workload="action-to-motion (15-layer denoiser, ActorVae 6 layers) B=512 total, 50 DDIM steps, decode 60x150"),
    "novae1024": dict(
        metric="motions/sec @ 1000-step DDPM raw-motion diffusion, batch 1024 over 8 GPUs", B=128, S=1, T=196, steps=1000,
        total_fixed=False, flop_per_motion=20.18e12, cpu_sample=1,
        workload="no-VAE raw-motion diffusion (trans_dec d=512) B=128/GPU (1024 over 8), 196x263, 1000 DDPM steps, CFG 7.5"),
}


# what the timed path returns per workload (--dump-outputs file name)
OUTPUT_NAME = {"headline": "joints", "1prompt": "joints", "action512": "feats", "novae1024": "motion"}
DUMP_LIMIT = 64_000_000      # bytes per dump; a larger output is sampled along its batch dimension


def dump_output(path: str, name: str, out, batch_dim: int):
    """``out`` as float32 ``path/<name>.npy``.  When it exceeds DUMP_LIMIT, a fixed seeded sample of motions
    along ``batch_dim`` (the same rows for the same shape in every run)."""
    import numpy as np
    import torch
    n = out.shape[batch_dim]
    keep = min(n, (DUMP_LIMIT - 4096) // (out.numel() // n * 4))          # 4 KB for the .npy header
    if keep < n:
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        out = out.index_select(batch_dim, rows.to(out.device))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"{name}.npy"), out.float().cpu().numpy())
    _log(f"dumped {name} {list(out.shape)} ({keep} of {n} motions) to {path}")


def _cpu_threads() -> int:
    # torch's intra-op pool on hundreds of threads thrashes on these small GEMMs; cap it
    return max(1, min(os.cpu_count() or 1, 32))


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""

    def __init__(self, index: int = 0):
        self.rows, self._p, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap,power.limit")
        try:
            self._p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                        "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self._p = None

    def _read(self):
        for line in self._p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self._p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self._p.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        def col(i):
            out = []
            for r in self.rows:
                try:
                    out.append(float(r[i]))
                except (IndexError, ValueError):
                    pass
            return out
        pw, pl = col(2), col(7)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w": statistics.median(pw) if pw else None,
                "power_limit_w": max(pl) if pl else None}


# ------------------------------------------------------------------------------------ model setups
def build_case(name: str, device=None):
    """(engine factory, oracle runner factory, synthetic inputs) for a workload.  The oracle runner is the
    CPU / eager-GPU restatement of the SAME path on the same seeded weights and inputs."""
    import torch
    from mld_b200 import synth
    w = WORKLOADS[name]
    mean, std = synth.mean_std()
    if name in ("headline", "1prompt"):
        dsd, vsd = synth.denoiser_state_dict(1234), synth.mld_vae_state_dict(4321)
        cfg_kw = dict()

        def inputs(B, seed):
            return synth.text_context(B, w["S"], seed=1 + seed), synth.init_noise(B, seed=2 + seed), None

        def oracle_run(O, sds, ctx, noise, lengths, step_noise, mean_, std_, steps=w["steps"]):
            return O.mld_forward(sds[0], O.DenoiserCfg(), sds[1], O.VaeCfg(), O.DDIMScheduler(), steps, ctx, noise,
                                 lengths, mean_, std_)[0]
        sds = (dsd, vsd)
    elif name == "action512":
        dsd = synth.denoiser_state_dict(seed=2345, condition="action", num_layers=15, nclasses=12, nfeats=150)
        vsd = synth.actor_vae_state_dict(seed=777)
        cfg_kw = dict(condition="action", num_layers=15, nclasses=12, nfeats=150, vae="actor", vae_layers=6, vae_nfeats=150)
        mean, std = synth.mean_std(150)

        def inputs(B, seed):
            g = torch.Generator().manual_seed(1 + seed)
            actions = torch.randint(0, 12, (B, 1), generator=g)
            return torch.cat([torch.zeros_like(actions), actions]), synth.init_noise(B, seed=2 + seed), None

        def oracle_run(O, sds, cond, noise, lengths, step_noise, mean_, std_, steps=w["steps"]):
            acfg = O.DenoiserCfg(condition="action", num_layers=15, nclasses=12, nfeats=150)
            z = O.diffusion_reverse(sds[0], acfg, O.DDIMScheduler(), steps, cond, noise, lengths)
            return O.vae_decode(sds[1], O.VaeCfg(kind="actor", nfeats=150, num_layers=6), z, lengths)
        sds = (dsd, vsd)
    else:
        dsd = synth.denoiser_state_dict(seed=3456, arch="trans_dec", d=512, diffusion_only=True)
        cfg_kw = dict(arch="trans_dec", latent_dim=(1, 512), diffusion_only=True, vae="none", scheduler="ddpm")

        def inputs(B, seed):
            g = torch.Generator().manual_seed(2 + seed)
            return synth.text_context(B, 1, seed=1 + seed), torch.randn(B, w["T"], 263, generator=g), 100 + seed

        def oracle_run(O, sds, ctx, x0, lengths, step_noise, mean_, std_, steps=w["steps"]):
            cfg = O.DenoiserCfg(arch="trans_dec", latent_dim=512, diffusion_only=True)
            return O.diffusion_reverse(sds[0], cfg, O.DDPMScheduler(), steps, ctx, x0, lengths, step_noise=step_noise)
        sds = (dsd,)

    def make_engine(dev_index):
        from mld_b200.engine import Engine, make_config
        eng = Engine(make_config(**cfg_kw), dev_index)
        eng.load_state_dict(dsd, "denoiser.")
        if len(sds) > 1:
            eng.load_state_dict(sds[1], "vae.")
        eng.finalize()
        if name != "novae1024":
            eng.set_mean_std(mean, std)
        eng.set_timesteps(w["steps"])
        return eng
    return w, make_engine, oracle_run, inputs, sds, (mean, std)


def cpu_reference_sample(torch, name: str, B: int, threads: int):
    """One bounded sample of the workload on the host cores through the oracle (fp32, eval)."""
    from oracle import mld_oracle as O
    torch.set_num_threads(threads)
    w, _, oracle_run, inputs, sds, (mean, std) = build_case(name)
    cond, noise, nseed = inputs(B, 0)
    step_noise = None
    steps = run_steps = w["steps"]
    if name == "novae1024":          # 1000 DDPM steps of a 9-layer d=512 model on a CPU: time 10 steps, scale
        run_steps = 10
        g = torch.Generator().manual_seed(nseed)
        step_noise = torch.randn(run_steps, B, w["T"], 263, generator=g)

    def run():
        with torch.no_grad():
            t0 = time.perf_counter()
            oracle_run(O, sds, cond, noise, [w["T"]] * B, step_noise, mean, std, run_steps)
            return (time.perf_counter() - t0) * (steps / run_steps)      # scaled to the full number of steps
    return run


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    w = WORKLOADS[args.config]
    cores = _cpu_threads()
    nsample = max(w["cpu_sample"], 64) if args.config == "headline" else w["cpu_sample"]
    run = cpu_reference_sample(torch, args.config, nsample, cores)
    for _ in range(args.warmup):
        _log(f"reference warm-up: {run():.2f}s")
    times = []
    for _ in range(args.steps):
        times.append(run())
        _log(f"reference step: {times[-1]:.2f}s")
    total = sum(times)
    value = nsample * args.steps / total
    sample = (f"{nsample} motions per step of the workload (same shapes, weights and step count"
              + ("; 10 of the 1000 DDPM steps timed and scaled" if args.config == "novae1024" else "") + ")")
    print(json.dumps({
        "impl": "reference", "metric": w["metric"], "value": value,
        "unit": "motions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["workload"], "global_batch": w["B"] * (1 if w["total_fixed"] or args.scaling == "strong" else args.gpus),
                   "parallelism": "host threads", "weights": "random-init (seeded), reference architecture",
                   "cpu_sample_motions": nsample},
        "cpu_baseline": {"value": value, "unit": "motions/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "motions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ------------------------------------------------------------------------------------ eager-PyTorch-on-GPU baseline
def gpu_eager_baseline(torch, name, dev, eng_joints, cond_d, noise_d, lengths, B):
    """The reference path restated in eager PyTorch (the oracle port; /root/reference does not exist on this
    box) on the SAME B200: fp32 with TF32 off and on, CUDA-event timed, with the joint error of the TF32 run and
    of this library against the fp32 eager result."""
    from oracle import mld_oracle as O
    w, _, oracle_run, _, sds, (mean, std) = build_case(name)
    sds_d = tuple({k: v.to(dev) for k, v in sd.items()} for sd in sds)
    mean_d, std_d = mean.to(dev), std.to(dev)
    out = {}
    ref = None
    for tag, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.backends.cudnn.allow_tf32 = tf32

        def run():
            with torch.no_grad(), torch.device(dev):
                return oracle_run(O, sds_d, cond_d, noise_d, lengths, None, mean_d, std_d)
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 2
        e0.record()
        for _ in range(reps):
            res = run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        joints = torch.stack([r for r in res]) if isinstance(res, (list, tuple)) else res
        entry = {"motions_per_s": B / (ms * 1e-3), "ms_per_batch": ms}
        if ref is None:
            ref = joints
            if eng_joints is not None:
                err = max(float((eng_joints[b] - ref[b]).abs().max() / ref[b].abs().max()) for b in range(B))
                entry["this_library_joint_rel_err_vs_fp32_eager"] = err
        else:
            entry["joint_rel_err_vs_fp32_eager"] = max(
                float((joints[b] - ref[b]).abs().max() / ref[b].abs().max()) for b in range(B))
        out[tag] = entry
        _log(f"eager {tag}: {ms:.1f} ms/batch")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out["what"] = ("oracle port of the reference modules (same weights, inputs, 50 steps, decode, joints) in eager PyTorch "
                   f"{torch.__version__} on this GPU, B={B}")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the b200 path's result; the reference arm times a sample of the workload")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3) if args.config != "novae1024" else max(args.warmup, 1)

    import torch
    import torch.distributed as dist
    import __graft_entry__ as g
    g.build()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    name = args.config
    w, make_engine, oracle_run, inputs, sds, (mean, std) = build_case(name)
    strong = w["total_fixed"] or args.scaling == "strong"
    if strong and w["B"] % world:
        raise SystemExit(f"batch {w['B']} does not split over {world} GPUs")
    B = w["B"] // world if strong else w["B"]            # motions per GPU
    S, T, NS = w["S"], w["T"], w["steps"]
    eng = make_engine(local_rank)
    if world > 1:
        eng.comm_init()                                  # NCCL communicator inside the library (C ABI)
    _log("engine ready")

    lengths = [T] * B
    cond_h, noise_h, nseed = inputs(B, rank)
    cond_h, noise_h = cond_h.pin_memory(), noise_h.pin_memory()
    len_h = torch.tensor(lengths, dtype=torch.int32).pin_memory()
    cond_d, noise_d = cond_h.to(dev), noise_h.to(dev)
    latent_model = name != "novae1024"
    step_noise_d = None
    if not latent_model:                                 # per-step DDPM noise, seeded per rank, generated on the device
        gd = torch.Generator(device=dev).manual_seed(nseed)
        step_noise_d = torch.randn((NS, B, T, 263), generator=gd, device=dev)
    J = eng.cfg.njoints
    out_shape = (world * B, T, J, 3)
    joints_h = torch.empty(out_shape, dtype=torch.float32).pin_memory() if latent_model else None
    gathered = [torch.empty(out_shape, dtype=torch.float32, device=dev) for _ in range(2)] if latent_model else None

    class _L(list):     # lengths list with a cached max (avoids a sync per call)
        pass
    len_list = _L(lengths)
    flip = [0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    feats_all = None
    if name == "action512" and world > 1:
        feats_all = torch.empty((world * B, T, eng.cfg.vae_nfeats), dtype=torch.float32, device=dev)

    def step_device():
        if not latent_model:                             # raw-motion diffusion: the motion itself is the result
            z = eng.diffusion_reverse(cond_d, noise_d, len_list, step_noise=step_noise_d)
            return eng.allgather(z.permute(1, 0, 2).contiguous()) if world > 1 else z
        if name == "action512":                          # 150-feature HumanAct12 motions: the decoded feats are the result
            out = eng.sample(cond_d, noise_d, len_list, want=("feats",))["feats"]
            return eng.allgather(out, feats_all) if world > 1 else out
        if world == 1:
            return eng.sample(cond_d, noise_d, len_list, want=("joints",))["joints"]
        # the one collective of the path, through the C ABI, on a side stream: batch i's gather overlaps batch i+1
        flip[0] ^= 1
        return eng.sample_gather(cond_d, noise_d, len_list, T=T, out=gathered[flip[0]], wait=False)

    def step_e2e():
        if latent_model and name != "action512":
            eng.sample_host(cond_h, noise_h, len_h, joints_h, T)          # C-ABI call with HOST buffers (gathers when N > 1)
        else:
            c, z = cond_h.to(dev, non_blocking=True), noise_h.to(dev, non_blocking=True)
            if latent_model:
                out = eng.sample(c, z, len_list, want=("feats",))["feats"]
            else:
                out = eng.diffusion_reverse(c, z, len_list, step_noise=step_noise_d)
            e2e_out.copy_(out, non_blocking=True)

    e2e_out = None
    if name == "action512":
        e2e_out = torch.empty((B, T, eng.cfg.vae_nfeats), dtype=torch.float32).pin_memory()
    elif not latent_model:
        e2e_out = torch.empty((T, B, 263), dtype=torch.float32).pin_memory()

    def timed(fn, K, W):
        for _ in range(W):
            fn()
        if world > 1 and latent_model:
            eng.gather_wait()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.launch_count
        e0.record()
        for a, b in evs:
            a.record()
            out = fn()
            b.record()
        if world > 1 and latent_model:
            eng.gather_wait()                            # the last batch's gather is inside the timed region
        e1.record()
        barrier()
        total_ms = e0.elapsed_time(e1)
        per = [a.elapsed_time(b) for a, b in evs]
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)      # max over ranks
        return float(t.item()), per, eng.launch_count - l0, out

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    total_ms, per, launches, last = timed(step_device, args.steps, args.warmup)
    clk = clocks.stop() if rank == 0 else None
    _log(f"device-resident: {total_ms / args.steps:.1f} ms/step")
    if args.dump_outputs and rank == 0:
        # every path returns batch-first except raw-motion diffusion on one GPU ([T, B, 263])
        dump_output(args.dump_outputs, OUTPUT_NAME[name], last, 1 if not latent_model and world == 1 else 0)
    del last
    e2e_ms, _, _, _ = timed(step_e2e, args.steps, 1)
    _log(f"e2e: {e2e_ms / args.steps:.1f} ms/step")

    value = world * B * args.steps / (total_ms / 1e3)
    e2e_value = world * B * args.steps / (e2e_ms / 1e3)
    peaks, peak_src = _peaks()

    step_p50 = None
    roof = None
    if rank == 0 and name in ("headline", "1prompt"):
        try:
            ms = eng.profile_steps(cond_d, noise_d)
            step_p50 = statistics.median(ms)
            _log(f"DDIM step p50 {step_p50:.3f} ms (eager launches, events between steps)")
        except Exception as e:                           # noqa: BLE001
            _log(f"profile_steps failed: {e}")
    if rank == 0 and name == "headline":
        # dominant kernel: every operator of one encoder layer timed in isolation at the full-batch shape
        M = 2 * w["B"] * (1 + 1 + S) if not strong else 2 * B * (1 + 1 + S)
        Bp = M // (2 * (2 + S))
        ops = {"qkv": 2.0 * M * 256 * 768, "ffn": 2.0 * M * 256 * 1024 * 2,
               "outproj_ln": 2.0 * M * 256 * 256, "attn": 4.0 * M * (1 + 1 + S) * 256}
        kname = {"qkv": "k_gemm_tc<256,2,EPI_FAST> (QKV projection, N=768, K=256)",
                 "ffn": "k_ffn_tc<2> (fused FFN: N=1024 up + GELU, N=256 down + residual + LayerNorm)",
                 "outproj_ln": "k_gemm_tc<256,2,EPI_LN> (attention out-projection + residual + LayerNorm)",
                 "attn": "k_attn_tc<64> (tcgen05 attention)"}
        times = {}
        for k in ops:
            times[k] = eng.profile_op(k, Bp, S, 10)
            _log(f"op {k}: {times[k]:.3f} ms")
        layer_ms = eng.profile_op("layer", Bp, S, 5)
        dom = max(times, key=times.get)
        peak = peaks.get("bf16_tflops", 1590.0)
        achieved = ops[dom] / (times[dom] * 1e-3) / 1e12
        traffic, traffic_src = None, None
        for fn in ("r02_traffic.json", "r01_traffic.json"):
            try:
                with open(os.path.join(ROOT, "profiles", fn)) as f:
                    traffic = json.load(f).get(dom)
                traffic_src = f"static: ncu --set full capture of this kernel, profiles/{fn} (not re-measured in this run)"
                break
            except Exception:
                continue
        roof = {"bound": "tensor", "kernel": f"{kname[dom]}, M={M}",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src + " bf16 burst (MEASURED_PEAKS.json)" if peak_src == "measured" else peak_src,
                "note": "achieved = algorithmic 2*M*N*K per launch / CUDA-event time; the split-fp16 scheme issues 3 "
                        "tensor-core passes per algorithmic FLOP (tensor-pipe rate = 3x achieved)",
                "tensor_pass_tflops": 3 * achieved,
                "tensor_pass_frac_of_sustained": 3 * achieved / peaks.get("bf16_tflops_sustained", 1400.0),
                "op_ms": {k: round(v, 4) for k, v in times.items()}, "layer_ms": round(layer_ms, 4),
                "op_tflops": {k: round(ops[k] / (times[k] * 1e-3) / 1e12, 1) for k in ops},
                "path_tflops": w["flop_per_motion"] * value / 1e12,
                "path_frac_of_sustained": w["flop_per_motion"] * value / 1e12 / peaks.get("bf16_tflops_sustained", 1400.0)}
    elif rank == 0:
        roof = {"bound": "tensor" if name != "1prompt" else "hbm", "kernel": "whole path", "achieved": w["flop_per_motion"] * value / 1e12,
                "peak": peaks.get("bf16_tflops_sustained", 1400.0), "unit": "TFLOP/s",
                "frac": w["flop_per_motion"] * value / 1e12 / peaks.get("bf16_tflops_sustained", 1400.0), "traffic": None,
                "note": "whole-path algorithmic FLOP rate against the sustained bf16 peak (per-kernel rooflines: headline config)"}

    eager = None
    if rank == 0 and world == 1 and name in ("headline", "1prompt") and not args.no_eager_baseline:
        try:
            jo = eng.sample(cond_d, noise_d, len_list, want=("joints",))["joints"]
            eager = gpu_eager_baseline(torch, name, dev, jo, cond_d, noise_d, lengths, B)
            eager["e2e_speedup_over_fp32_eager"] = e2e_value / eager["fp32"]["motions_per_s"]
            eager["e2e_speedup_over_tf32_eager"] = e2e_value / eager["tf32"]["motions_per_s"]
        except Exception as e:                           # noqa: BLE001
            eager = {"error": f"{type(e).__name__}: {e}"}
            _log(f"eager baseline failed: {e}")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = _cpu_threads()
        nsample = w["cpu_sample"]
        _log(f"cpu baseline on {cores} threads, {nsample} motions")
        run = cpu_reference_sample(torch, name, nsample, cores)
        run()
        dt = min(run(), run())
        _log(f"cpu baseline: {dt:.2f}s per {nsample} motions")
        cpu = {"value": nsample / dt, "unit": "motions/s", "cores": cores, "kind": "port",
               "sample": f"{nsample} motions of the same workload (same shapes, weights and steps), best of 2 after 1 "
                         f"warm-up, oracle port pinned to the reference modules"}

    if rank == 0:
        h2d = cond_h.numel() * cond_h.element_size() + noise_h.numel() * 4 + len_h.numel() * 4
        d2h = (joints_h.numel() if joints_h is not None else e2e_out.numel()) * 4
        print(json.dumps({
            "metric": w["metric"], "value": value, "unit": "motions/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "ddim_step_p50_ms": step_p50, "batch_p50_ms": statistics.median(per), "higher_is_better": True,
            "scaling": "strong" if strong else "weak", "vs_baseline": None,
            "dtype": "f16x2-split (fp32-equivalent, fp32 accumulate)", "data": "synthetic",
            "config": {"workload": w["workload"], "global_batch": world * B, "parallelism": f"batch-sharded dp{world}",
                       "l2": "working set (activations > 700 MB at B=256) exceeds the 126 MB L2; no flush needed" if name == "headline"
                             else "inputs + weights smaller than L2: steady-state (warm L2) numbers, as in the real loop",
                       "weights": "random-init (seeded), reference architecture"},
            "e2e": {"value": e2e_value, "unit": "motions/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk, "roofline": roof, "cpu_baseline": cpu, "gpu_eager_baseline": eager,
            "kernel_stats": eng.kernel_stats(),
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
