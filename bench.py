#!/usr/bin/env python
"""Headline benchmark: mel-frames/sec of the Grad-TTS reverse-diffusion sampler at N=50 steps.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the mel the timed path returned in its last timed step as DIR/mel.npy (float32).  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.

One bench "step" = one full `Diffusion.forward(z, mask, mu, n_timesteps=50)` call on the workload
BASELINE.json quotes the metric on (config 2: B=32 utterances x T=512 frames, fp32 in/out, per GPU;
weak scaling: every rank samples its own 32 utterances, outputs all-gathered).  Prints ONE JSON line.

  value        frames/s, inputs resident in HBM, CUDA-event timed, max over ranks
  e2e          same metric through the host-buffer entry point (pinned host tensors in/out, copies timed)
  roofline     the dominant kernel class (3x3 conv implicit GEMMs), timed per launch with CUDA events
  cpu_baseline the CPU oracle (a port of the reference's PyTorch path) on a bounded sample, this box's cores
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
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree: leave no __pycache__ behind

WORKLOADS = {
    # BASELINE.json configs[1]: Grad-TTS batch=32, T~512, N=50, fp32, 1xB200
    "gradtts_b32_t512_n50": dict(B=32, T=512, N=50, n_spks=1),
    # BASELINE.json configs[4]'s per-GPU share (2048 utterances over 8 GPUs = 256 per GPU); not the default bench line:
    #   torchrun --nproc-per-node 8 bench.py --gpus 8 --workload gradtts_b256_t512_n50 --steps 2 --warmup 3 --no-fp32-leg
    "gradtts_b256_t512_n50": dict(B=256, T=512, N=50, n_spks=1),
}
FLOP_PER_FRAME_STEP = 134.15e6      # SURVEY.md 8(d): 67,077,120 MAC per mel frame per reverse step
IDEAL_BYTES_PER_FRAME_STEP = 713280.0
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each tensor of `arrays` as <out_dir>/<name>.npy in float32, DUMP_MAX_BYTES in all.  A tensor over its share
    keeps a fixed, seeded sample of its utterances (dim 0), the same rows in every run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_MAX_BYTES // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > share:
            rows = np.random.default_rng(0).choice(a.shape[0], share // (a.nbytes // a.shape[0]), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float32))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, bf16=1400.0, src="fallback")


def measure_tf32_matmul_tflops(torch, dev, seconds=1.0):
    """Sustained cuBLAS TF32 rate on this GPU (torch.matmul 8192^3, fp32 tensors, allow_tf32), back to back for
    `seconds`: MEASURED_PEAKS.json only carries the bf16 rate, and tf32 is not exactly half of it in practice."""
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters, t0 = 0, time.perf_counter()
        e0.record()
        while True:
            for _ in range(10):
                a @ b
            iters += 10
            torch.cuda.synchronize()
            if time.perf_counter() - t0 > seconds:
                break
        e1.record()
        torch.cuda.synchronize()
        return 2.0 * n ** 3 * iters / (e0.elapsed_time(e1) * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.lines, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(dev)], stdout=subprocess.PIPE, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.th.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def _ncpu():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count()


# ---- the CPU arm: the UNMODIFIED reference (oracle/_ref bytecode or /root/reference) when present, else the oracle port ------
CPU_SAMPLE_B = 8          # utterances of the workload's T per timed sample (VERDICT r1: B >= 8, >= 3 Euler steps, not extrapolated from B=2)
CPU_SAMPLE_STEPS = 3
_CPU = {}


def _cpu_runner(wl, torch):
    """Build once: (fn(z, mask, mu, n_steps, spk) -> mel, kind, description).  The reference's own `Diffusion` module
    (Grad-TTS/model/diffusion.py:227-279) with the bench's synthetic weights loaded strictly, run on the host cores."""
    if "fn" in _CPU:
        return _CPU["fn"], _CPU["kind"], _CPU["what"]
    from oracle import ref_import
    from speech_backbones_b200 import UNetConfig, synthetic_state_dict
    cfg = UNetConfig(n_spks=wl["n_spks"])
    sd = synthetic_state_dict(cfg)
    if ref_import.available("gradtts"):
        md = ref_import.import_model("gradtts")
        dec = md.Diffusion(cfg.n_feats, cfg.dim, n_spks=cfg.n_spks, spk_emb_dim=cfg.spk_emb_dim).eval()
        dec.load_state_dict(sd, strict=True)

        def fn(z, mask, mu, n, spk):
            return dec(z, mask, mu, n, False, spk)
        kind, what = "reference", f"unmodified reference Diffusion.forward ({ref_import.kind('gradtts')})"
    else:
        from oracle import gradtts_oracle as O

        def fn(z, mask, mu, n, spk):
            return O.reverse_diffusion(sd, cfg, z, mask, mu, n, False, spk)
        kind, what = "port", "oracle port of the reference (oracle/gradtts_oracle.py; oracle/_ref not built)"
    _CPU.update(fn=fn, kind=kind, what=what, cfg=cfg)
    return fn, kind, what


def pick_cpu_threads(torch, fn, inputs):
    """The CPU arm gets all the host threads it can USE: the thread count is swept AT THE SAMPLE'S OWN SHAPE (one Euler
    step each, after one untimed step) up to every usable core, and the fastest is kept (PyTorch's CPU convs slow down
    when oversubscribed on many-core boxes)."""
    if "threads" in _CPU:
        torch.set_num_threads(_CPU["threads"])
        return _CPU["threads"], _CPU["sweep"]
    z, mask, mu, spk = inputs
    n = _ncpu()
    cands = sorted({c for c in (8, 16, 32, 48, 64, 96, 128, n) if c <= n})
    sweep, best, best_t = {}, cands[0], float("inf")
    torch.set_num_threads(cands[0])
    fn(z, mask, mu, 1, spk)                                                      # page in / allocator warm-up
    for c in cands:
        torch.set_num_threads(c)
        fn(z, mask, mu, 1, spk)
        t0 = time.perf_counter()
        fn(z, mask, mu, 1, spk)
        dt = time.perf_counter() - t0
        sweep[c] = round(dt, 3)
        if dt < best_t:
            best, best_t = c, dt
        elif dt > 1.5 * best_t:
            break                                                               # oversubscribed: larger counts only get slower
    _CPU.update(threads=best, sweep=sweep)
    torch.set_num_threads(best)
    return best, sweep


def cpu_reference_sample(wl, torch):
    """ONE sample definition for both the `--impl reference` arm and the `cpu_baseline` leg: CPU_SAMPLE_B utterances at the
    workload's T for CPU_SAMPLE_STEPS Euler steps (one call of the reference's `Diffusion.forward` with n_timesteps =
    CPU_SAMPLE_STEPS; the loop body is step-independent, diffusion.py:258-274), timed in full, after a warm-up call.
    mel-frames/s at the workload's N = frames / (seconds per frame-step x N)."""
    from speech_backbones_b200 import synthetic_inputs
    fn, kind, what = _cpu_runner(wl, torch)
    b, n_steps = min(CPU_SAMPLE_B, wl["B"]), CPU_SAMPLE_STEPS
    z, mask, mu, spk, _ = synthetic_inputs(b, wl["T"], n_spks=wl["n_spks"])
    with torch.no_grad():
        threads, sweep = pick_cpu_threads(torch, fn, (z, mask, mu, spk))
        t0 = time.perf_counter()
        y = fn(z, mask, mu, n_steps, spk)
        dt = time.perf_counter() - t0
    assert torch.isfinite(y).all()
    sec_per_frame_step = dt / (b * wl["T"] * n_steps)
    frames_per_sec = 1.0 / (sec_per_frame_step * wl["N"])
    sample = (f"{what}, PyTorch CPU fp32, {threads} threads (fastest of a sweep at this shape: {sweep} s per Euler step; "
              f"{_ncpu()} usable cores); B={b} x T={wl['T']}, {n_steps} Euler steps timed in full ({dt:.2f} s); "
              f"mel-frames/s at N={wl['N']} = B*T / (s per step * N)")
    return frames_per_sec, sec_per_frame_step, sample, threads, kind, y


def run_reference(args, wl):
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals = []
    for i in range(args.warmup + args.steps):
        fps, spfs, sample, threads, kind, y = cpu_reference_sample(wl, torch)
        if i >= args.warmup:
            vals.append((fps, spfs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"mel": y})
    fps = statistics.median(v[0] for v in vals)
    ms_full = statistics.median(v[1] for v in vals) * wl["B"] * wl["T"] * wl["N"] * 1e3
    out = {
        "impl": "reference", "metric": "mel-frames/sec at N=50 reverse-diffusion steps", "value": fps,
        "unit": "mel-frames/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_full, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, wl, int(os.environ.get("WORLD_SIZE", "1")),
                               note="CPU reference arm: each bench step is one bounded sample (see cpu_baseline.sample); "
                                    "ms_per_step is that rate applied to the full workload"),
        "cpu_baseline": {"value": fps, "unit": "mel-frames/s", "cores": threads, "kind": kind, "sample": sample,
                         "spread": {"min": min(v[0] for v in vals), "max": max(v[0] for v in vals), "n": len(vals)}},
        "e2e": {"value": fps, "unit": "mel-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def bench_config(args, wl, world, **extra):
    """The `config` object: identical keys in both arms (the driver compares them)."""
    cfg = {"workload": args.workload, "batch_per_gpu": wl["B"], "global_batch": wl["B"] * world, "frames": wl["T"],
           "n_timesteps": wl["N"], "stoc": False, "parallelism": f"dp{world}"}
    cfg.update(extra)
    return cfg


# per-mode arithmetic + the parity bound its tests hold it to (tests/test_fp32x3_gpu.py, tests/test_parity_gpu.py)
MODES = {
    "fp32x3": dict(dtype="f32", what="fp32-class on tcgen05: x*w = x_hi*w_hi (kind::tf32) + (x_lo*w + x*w_lo) as one kind::f16 MMA over packed "
                                     "fp16 correction chunks, fp32 accumulate with runs folded in fp32; exact fp32 GN/Mish/softmax/Euler",
                   tol="rel-L2 <= 1e-5 per estimator call vs the reference's fp32 CPU outputs (13 goldens; measured 2.2-2.9e-6), <= 2e-4 on N<=50 trajectories (measured 1.1-1.4e-6)",
                   mma_per_mac=2),
    "tf32": dict(dtype="tf32", what="tcgen05 kind::tf32 operands (PyTorch's default GPU conv arithmetic), fp32 accumulate / GN / softmax / Euler",
                 tol="rel-L2 <= 4e-3 per estimator call (measured 1.5e-3), <= 8e-3 on trajectories", mma_per_mac=1),
    "bf16": dict(dtype="bf16", what="bf16 operand tensors + weights on tcgen05 kind::f16 (BASELINE config 3's arithmetic), fp32 accumulate / GN / state",
                 tol="rel-L2 <= 2e-2 per estimator call (measured 1.1e-2), <= 1e-2 on trajectories", mma_per_mac=1),
    "fp32": dict(dtype="f32", what="CUDA-core FFMA implicit GEMM (the round-1 exact mode; kept as a second opinion)",
                 tol="rel-L2 <= 1e-4 per estimator call (measured 0.6-2.6e-6)", mma_per_mac=0),
}


def csrc_digest():
    """sha256 over the kernel sources: ties measured side files (profiles/r2_traffic_*.json) to the binary being benched."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "speech-backbones_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".h")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the sampler has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    from speech_backbones_b200 import UNetConfig, estimator_param_spec, synthetic_inputs, synthetic_state_dict
    from speech_backbones_b200.gradtts import Diffusion
    from speech_backbones_b200.sharded import broadcast_state_dict, sharded_sample

    B, T, N = wl["B"], wl["T"], wl["N"]
    cfg = UNetConfig(n_spks=wl["n_spks"])
    # weights: rank 0 owns them, NCCL broadcast to the other ranks (north_star: weight broadcast + mel gather only)
    t0 = time.perf_counter()
    sd = synthetic_state_dict(cfg) if rank == 0 else None
    if world > 1:
        sd = broadcast_state_dict(sd, estimator_param_spec(cfg), dev)
        torch.cuda.synchronize()
    bcast_s = time.perf_counter() - t0

    z, mask, mu, spk, _ = synthetic_inputs(B, T, seed=1234 + rank, n_spks=cfg.n_spks)
    zd, md, mud = z.to(dev), mask.to(dev), mu.to(dev)
    spd = None if spk is None else spk.to(dev)
    gathered = torch.empty((world * B, cfg.n_feats, T), dtype=torch.float32, device=dev) if world > 1 else None

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make(precision):
        d = Diffusion(cfg.n_feats, cfg.dim, n_spks=cfg.n_spks, precision=precision).eval()
        d.load_state_dict(sd)
        return d.to(dev)

    def time_mode(dec_, steps, warmup, sample_clocks=False):
        """W untimed + K timed `Diffusion.forward` calls (+ the output all-gather when world > 1), CUDA events on the
        launching stream, barrier + synchronize on both sides, MAX over ranks.  Also times the gather alone per call."""
        eng_ = dec_.engine()
        y = None
        for _ in range(warmup):
            y = dec_(zd, md, mud, N, False, spd)
            if world > 1:
                dist.all_gather_into_tensor(gathered, y)
        fence()
        clocks = ClockSampler(local) if (sample_clocks and rank == 0) else None
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps + 2)]
        launches = 0
        ev[0].record()
        for i in range(steps):
            y = dec_(zd, md, mud, N, False, spd)
            launches += eng_.last_launch_count()
            ev[1 + 2 * i].record()
            if world > 1:
                dist.all_gather_into_tensor(gathered, y)       # output mel gather over NVLink
            ev[2 + 2 * i].record()
        ev[2 * steps + 1].record()
        fence()
        clk = clocks.stop() if clocks else None
        ms_total = ev[0].elapsed_time(ev[2 * steps + 1])
        gather_ms = sum(ev[1 + 2 * i].elapsed_time(ev[2 + 2 * i]) for i in range(steps)) / steps
        tms = torch.tensor([ms_total, gather_ms], dtype=torch.float64, device=dev)
        per_rank = None
        if world > 1:
            allr = [torch.zeros_like(tms) for _ in range(world)]
            dist.all_gather(allr, tms)
            per_rank = [{"rank": r, "ms_per_step": round(v[0].item() / steps, 3), "gather_ms": round(v[1].item(), 3)} for r, v in enumerate(allr)]
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms_step = tms[0].item() / steps
        return dict(ms_step=ms_step, value=world * B * T / (ms_step * 1e-3), launches=launches, clocks=clk, y=y,
                    per_rank=per_rank, gather_ms_max=tms[1].item())

    dec = make(args.precision)
    eng = dec.engine()
    head = time_mode(dec, args.steps, args.warmup, sample_clocks=True)
    ms_step, value, launches, clk = head["ms_step"], head["value"], head["launches"], head["clocks"]
    # what a caller of the timed path receives from its last step: the mel, all-gathered over the ranks when world > 1
    head_out = (gathered.clone() if world > 1 else head["y"]) if args.dump_outputs else None

    # ---- end to end through the host-buffer entry point (pinned host memory in/out, copies inside the timed region)
    zh, mh, muh = z.pin_memory(), mask.pin_memory(), mu.pin_memory()
    outh = torch.empty_like(z).pin_memory()
    sph = None if spk is None else spk.pin_memory()
    eng.reverse_diffusion_host(zh, mh, muh, N, False, sph, None, outh)          # warm-up
    fence()
    t0 = time.perf_counter()
    e2e_steps = max(1, min(args.steps, 3))
    for _ in range(e2e_steps):
        eng.reverse_diffusion_host(zh, mh, muh, N, False, sph, None, outh)
        _ = float(outh[0, 0, 0])                                               # host read of the result
    fence()
    te = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * T / te.item()
    h2d = (zh.numel() + mh.numel() + muh.numel() + (0 if sph is None else sph.numel())) * 4
    d2h = outh.numel() * 4

    # ---- BASELINE config 5 as written (2048 utterances = 256 per GPU over 8 GPUs) through sharded.sharded_sample over NCCL
    config5 = None
    if (world == 8 or args.force_config5) and world > 1 and not args.no_config5:
        B5 = 256
        z5, m5, mu5, _, _ = synthetic_inputs(B5 * world, T, seed=4321, n_spks=1) if rank == 0 else (None,) * 5
        shape5 = (B5 * world, cfg.n_feats, T)
        ins = []
        for t_, shp in ((z5, shape5), (m5, (B5 * world, 1, T)), (mu5, shape5)):
            buf = t_.to(dev) if rank == 0 else torch.empty(shp, dtype=torch.float32, device=dev)
            dist.broadcast(buf, 0)
            ins.append(buf)
        del z5, m5, mu5

        def compute(zs, ms, mus, n, spk_):
            return dec(zs, ms, mus, n, False, None)
        sharded_sample(compute, ins[0], ins[1], ins[2], N)                     # warm-up (plan + graphs for B=256)
        fence()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        y5 = sharded_sample(compute, ins[0], ins[1], ins[2], N)
        c1.record()
        fence()
        t5 = torch.tensor([c0.elapsed_time(c1)], dtype=torch.float64, device=dev)
        all5 = [torch.zeros_like(t5) for _ in range(world)]
        dist.all_gather(all5, t5)
        dist.all_reduce(t5, op=dist.ReduceOp.MAX)
        config5 = {"workload": "BASELINE config 5: 2048 utterances x T=512, N=50, 256 per GPU, sharded_sample over NCCL (1 timed call)",
                   "value": B5 * world * T / (t5.item() * 1e-3), "unit": "mel-frames/s", "ms": t5.item(),
                   "per_rank_ms": [round(v.item(), 2) for v in all5], "finite": bool(torch.isfinite(y5).all().item()),
                   "gathered_shape": list(y5.shape)}
        del ins, y5

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel class, one CUDA event pair per launch
    peaks = load_peaks()
    mode = MODES[args.precision]
    dec(zd, md, mud, 1, False, spd)                                            # (config 5 may have re-planned for B=256)
    prof = eng.profile_ops()
    conv = [(n, ms, fl, by) for n, ms, fl, by in prof if n.endswith(".raw")]
    conv_ms, conv_fl, conv_by = (sum(x[i] for x in conv) for i in (1, 2, 3))
    all_ms = sum(x[1] for x in prof)
    # bf16 operands: the measured cuBLAS bf16 rate of MEASURED_PEAKS.json.  tf32 / fp32x3: that file has no tf32 figure, so
    # the tf32 rate is the larger of half the bf16 rate and a cuBLAS TF32 matmul timed here (sustained, ~1 s); an fp32x3
    # MAC costs two tensor-core passes at the tf32 instruction rate (one tf32 MMA + one fp16 correction MMA whose K = 16
    # covers x_lo*w and x*w_lo of the same 8 channels), so its algorithmic peak is half of that
    tf32_here = measure_tf32_matmul_tflops(torch, dev) if args.precision != "bf16" else None
    mma_peak = peaks["bf16"] if args.precision == "bf16" else max(peaks["bf16"] * 0.5, tf32_here)
    per_mac = max(1, mode["mma_per_mac"])
    tensor_peak = mma_peak / per_mac
    achieved = conv_fl / (conv_ms * 1e-3) / 1e12
    by_kind = {}
    for n, ms, fl, by in prof:
        k = ("conv3x3" if n.endswith(".raw") else "gn_mish_act" if n.endswith(".act") else
             "attention" if (".2." in n or "mid_attn" in n) else "resample" if ".3." in n else
             "final_euler" if n == "estimator.out" else "resblock_tail")
        by_kind[k] = by_kind.get(k, 0.0) + ms
    # DRAM bytes per launch of the same kernel class from an ncu capture OF THIS BINARY (scripts/ncu_traffic.py writes the
    # csrc digest next to the bytes); a capture of other kernels is not reported
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", f"r2_traffic_conv3x3_{args.precision}.json")
    if os.path.exists(tpath) and (B, T) == (32, 512):
        tj = json.load(open(tpath))
        if tj.get("csrc_digest") == csrc_digest():
            traffic, traffic_src = tj["dram_bytes_per_launch"], f"profiles/{os.path.basename(tpath)} (ncu dram__bytes_read+write, {tj['launches']} launches, csrc {tj['csrc_digest']})"
        else:
            traffic_src = f"not reported: profiles/{os.path.basename(tpath)} was captured from other kernel sources (csrc {tj.get('csrc_digest')} != {csrc_digest()})"
    roofline = {
        "kernel": "conv3x3 implicit GEMM (25 launches/step)", "bound": "tensor", "achieved": achieved, "peak": tensor_peak,
        "unit": "TFLOP/s", "frac": achieved / tensor_peak, "traffic": traffic, "traffic_source": traffic_src,
        "algorithmic_bytes_per_launch": conv_by / max(1, len(conv)),
        "traffic_note": ("fp32x3 reads every conv input twice by design (the fp32 tensor + its 16-byte-per-4-channels correction "
                         "chunks): expected DRAM bytes = algorithmic (4 B in + 4 B out per element) + the input bytes once more"
                         if args.precision == "fp32x3" else None),
        "peak_note": (f"{peaks['src']} cuBLAS bf16 sustained (MEASURED_PEAKS.json)" if args.precision == "bf16" else
                      f"tf32 MMA rate = max(0.5 x {peaks['src']} cuBLAS bf16 sustained = {peaks['bf16'] * 0.5:.1f}, cuBLAS TF32 matmul 8192^3 "
                      f"sustained measured in this run = {tf32_here:.1f}) TFLOP/s, divided by {per_mac} tensor-core pass(es) at the tf32 instruction rate per algorithmic MAC in mode {args.precision}"),
        "mma_issue_tflops": achieved * per_mac,
        "launches": len(conv), "avg_launch_ms": conv_ms / max(1, len(conv)),
        "flop_per_launch_avg": conv_fl / max(1, len(conv)), "share_of_step": conv_ms / all_ms,
        "hbm": {"achieved_gbs": conv_by / (conv_ms * 1e-3) / 1e9, "peak_gbs": peaks["hbm_gbs"],
                "frac": conv_by / (conv_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]},
        "step_ms_by_kind": {k: round(v, 4) for k, v in by_kind.items()},
        "whole_step": {"tflops": FLOP_PER_FRAME_STEP * B * T / (ms_step / N * 1e-3) / 1e12,
                       "frac_of_tensor_peak": FLOP_PER_FRAME_STEP * B * T / (ms_step / N * 1e-3) / 1e12 / tensor_peak,
                       "ideal_hbm_gbs": IDEAL_BYTES_PER_FRAME_STEP * B * T / (ms_step / N * 1e-3) / 1e9},
    }
    # ---- the other precision modes of the same engine, timed with the SAME --steps / --warmup (first-class legs)
    legs = {}
    if world == 1 and not args.no_extra_legs:
        y_head = head["y"]
        for prec in [m for m in ("fp32x3", "tf32", "bf16") if m != args.precision]:
            d2 = make(prec)
            r = time_mode(d2, args.steps, args.warmup)
            legs[prec] = {"value": r["value"], "unit": "mel-frames/s", "ms_per_step": r["ms_step"], "dtype": MODES[prec]["dtype"],
                          "steps": args.steps, "warmup": args.warmup, "arithmetic": MODES[prec]["what"], "tolerance": MODES[prec]["tol"],
                          "rel_l2_of_output_vs_headline_mode": ((r["y"] - y_head).double().norm() / y_head.double().norm()).item()}
            d2._engine.close()
            del d2, r
            torch.cuda.empty_cache()
    cpu = cpu_reference_sample(wl, torch) if world == 1 else None
    out = {
        "metric": "mel-frames/sec at N=50 reverse-diffusion steps", "value": value, "unit": "mel-frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": mode["dtype"], "data": "synthetic",
        "config": bench_config(args, wl, world, precision_mode=args.precision, arithmetic=mode["what"], tolerance=mode["tol"],
                               l2=f"per-step working set ({eng.workspace_bytes(B, T) / 1e9:.1f} GB of activations) exceeds the 126 MB L2; no flush needed",
                               weights="synthetic seeded (no checkpoints ship with the reference)",
                               weight_broadcast_s=round(bcast_s, 4)),
        "frame_steps_per_s": value * N,
        "e2e": {"value": e2e_value, "unit": "mel-frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches,
        "clocks": clk,
        "roofline": roofline,
    }
    if legs:
        out["modes"] = legs
    if head["per_rank"] is not None:
        out["per_rank"] = head["per_rank"]
        out["gather_ms_max"] = head["gather_ms_max"]
    if config5 is not None:
        out["config5"] = config5
    if cpu is not None:
        fps_cpu, _, sample, threads, kind, _ = cpu
        out["cpu_baseline"] = {"value": fps_cpu, "unit": "mel-frames/s", "cores": threads, "kind": kind, "sample": sample}
    if head_out is not None:
        dump_outputs(args.dump_outputs, {"mel": head_out})
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="gradtts_b32_t512_n50", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp32x3", choices=["fp32x3", "fp32", "tf32", "bf16"],
                    help="fp32x3 (default, the headline: BASELINE config 2 is fp32): fp32-class arithmetic on tcgen05 (tf32 + fp16 correction); "
                         "tf32: plain tf32 operands (PyTorch's default GPU conv arithmetic); bf16: bf16 operand tensors "
                         "(BASELINE config 3's arithmetic); fp32: the CUDA-core FFMA path")
    ap.add_argument("--no-extra-legs", "--no-fp32-leg", dest="no_extra_legs", action="store_true",
                    help="skip the other precision modes' legs (each is timed with the same --steps/--warmup)")
    ap.add_argument("--no-config5", action="store_true", help="at 8 GPUs: skip the BASELINE config 5 leg (B=256 per GPU)")
    ap.add_argument("--force-config5", action="store_true", help="run the config 5 leg (256 utterances per GPU) at any world size > 1 (debug)")
    ap.add_argument("--batch", type=int, default=None, help="override B (debug only; not a valid bench line)")
    ap.add_argument("--frames", type=int, default=None, help="override T (debug only)")
    ap.add_argument("--n-timesteps", type=int, default=None, help="override N (debug only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the mel the timed path returned in its last step as DIR/mel.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    wl = dict(WORKLOADS[args.workload])
    if args.batch: wl["B"] = args.batch
    if args.frames: wl["T"] = args.frames
    if args.n_timesteps: wl["N"] = args.n_timesteps
    if args.impl == "reference":
        run_reference(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
