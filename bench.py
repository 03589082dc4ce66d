#!/usr/bin/env python
"""Benchmark of the Panacea denoising hot path on B200 (BASELINE.json metric: UNet denoise-steps/s).

A "step" = one Euler/DDIM step of one 6-view x 8-frame sequence: CFG-doubled eps evaluation (ControlNet + UNet on
16 frames of [8, 32, 6x56]) + guidance + update — BASELINE.json configs[1] ("single-GPU 50-step DDIM, 6 views x 8
frames, synthetic BEV layout via ControlNet, bf16"). One sequence per GPU (weak scaling), no collective inside
the loop; after the loop rank 0 gathers the final latents over NCCL (configs[2]).

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
  python bench.py --impl reference [--steps K] [--warmup W]      # the reference algorithm on the host CPU (oracle port)
  python bench.py --steps K --dump-outputs DIR                    # also write the last timed step's outputs (rank 0)

Prints ONE JSON line (rank 0). Weights and inputs are fixed by the rank's seed, so two builds run with the same arguments
can be compared output for output: DIR/latent.npy is the latent after the last timed step ([8, 4, 32, 336], float32) and
DIR/eps.npy that step's CFG-doubled network output ([16, 4, 32, 336], float32).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

METRIC = "UNet denoise-steps/s (6-view x 8-frame latent, CFG-doubled eps-eval + guidance + Euler update)"
H, W_VIEW, VIEWS, T = 32, 56, 6, 8
ALGO_TFLOP_PER_STEP = 82.2        # SURVEY.md section 8d: steady-state algorithmic work of one CFG step at 32x56


_T0 = time.time()


def log(msg: str) -> None:
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


def workload_config(n_gpus: int) -> dict:
    return {"workload": "configs[1]: 50-step Euler/DDIM denoising loop, 1 sequence/GPU, 6 views x 8 frames, latent 32x56 per "
                        "view (x [16,8,32,336] per eps-eval incl. CFG), synthetic BEV hint [8,19,256,2688] + text [1,77,1024], "
                        "full-size UNet+ControlNet (2.24 B params, random init, zero-init tails re-drawn N(0,0.02^2))",
            "cfg_scale": 5.0, "frames": T, "views": VIEWS, "latent_hw_per_view": [H, W_VIEW],
            "sequences_per_gpu": 1, "parallelism": f"dp{n_gpus} (independent sequences, NCCL gather of final latents)",
            "l2_policy": "no explicit flush: every step streams 4.5 GB of bf16 weights + >2 GB of activations, >> 126 MB L2"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.samples, self.proc, self.thread = [], None, None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 7:
                self.samples.append(parts)

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for p in self.samples:
            try:
                sm.append(float(p[0])); mx = float(p[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU baseline (oracle)
def usable_cores() -> int:
    """Cores this process may really use: affinity mask, cgroup CPU quota, PN_CPU_THREADS override. (nproc can report
    128 on a box whose container is throttled to a fraction of that; running 128 OpenMP threads there is far slower
    than running 16.)"""
    if os.environ.get("PN_CPU_THREADS"):
        return max(1, int(os.environ["PN_CPU_THREADS"]))
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, 32))       # the op mix (thousands of small ops per eval) stops scaling well before 32 threads


def cpu_baseline(budget_s: float):
    """Times the CPU oracle port (oracle/unet_port.py — the reference algorithm restated in plain PyTorch fp32) on the
    host cores on REAL full-frame samples of the workload (BASELINE.md section 3), independent of --steps:
      A. always: one eps-eval of the full model on one full frame, x [1,8,32,336] (T=1, b=1; BASELINE config 1 shape);
      B. when the remaining budget allows (predicted from A with the survey's measured T=8/T=1 ratio of 4.0): one CFG
         half of the benchmarked step, x [8,8,32,336] (T=8, b=1) — a denoise step is exactly two of these.
    steps/s = 1 / (2 t_B) when B ran, else 1 / (16 t_A) (a step evaluates 16 frames; the T=8 batching gain is then NOT
    credited to the CPU). Returns (steps_per_s, description, cores, dict of measured seconds)."""
    from oracle import unet_port as P
    cores = usable_cores()
    torch.set_num_threads(cores)
    t_start = time.perf_counter()
    cfg = P.NetConfig()
    spec = P.state_spec(cfg)
    # cheap non-degenerate weights (timing only): tile one random block, scale like the seeded init
    g = torch.Generator().manual_seed(0)
    pool = torch.randn(1 << 22, generator=g)
    sd = {}
    for k, shape in spec.items():
        n = math.prod(shape)
        v = pool[:n] if n <= pool.numel() else pool.repeat((n + pool.numel() - 1) // pool.numel())[:n]
        v = v.reshape(shape)
        if k.endswith(".bias"):
            v = v * 0.05
        elif len(shape) == 1:
            v = 1.0 + 0.1 * v
        else:
            v = v * (0.7 / math.sqrt(math.prod(shape[1:])))
        sd[k] = v.contiguous()
    log(f"cpu baseline: weights ready after {time.perf_counter() - t_start:.1f}s, {cores} threads")

    def run(frames_T: int, b: int):
        c = P.NetConfig(num_frames=frames_T)
        BT, Wt = b * frames_T, VIEWS * W_VIEW
        x = torch.randn(BT, 4, H, Wt)
        cond = {"concat": torch.randn(BT, 4, H, Wt), "cond_feat": torch.rand(BT, 19, 8 * H, 8 * Wt), "crossattn": torch.randn(b, 77, 1024)}
        t = torch.full((BT,), 500, dtype=torch.int64)
        t0 = time.perf_counter()
        P.wrapper_forward(sd, c, x, t, cond)
        return time.perf_counter() - t0

    secs = {}
    secs["t1_full_frame_[1,8,32,336]"] = tA = run(1, 1)
    log(f"cpu baseline: full-frame T=1 eval {tA:.1f}s")
    remaining = budget_s - (time.perf_counter() - t_start)
    if 4.0 * tA * 1.15 <= remaining:
        secs["t8_cfg_half_[8,8,32,336]"] = tB = run(T, 1)
        log(f"cpu baseline: T=8 CFG-half eval {tB:.1f}s")
        val = 1.0 / (2.0 * tB)
        desc = (f"measured: one CFG half x[8,8,32,336] (T=8, b=1) in {tB:.1f} s -> step = 2 halves; also one full frame "
                f"x[1,8,32,336] in {tA:.1f} s")
    else:
        val = 1.0 / (16.0 * tA)
        desc = (f"measured: one full frame x[1,8,32,336] (T=1, b=1) in {tA:.1f} s -> step = 16 frame-evals (the T=8 CFG half "
                f"did not fit the {budget_s:.0f} s budget)")
    return val, f"{desc}; oracle port, torch {torch.__version__} fp32, {cores} threads (nproc {os.cpu_count()})", cores, secs


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = float(os.environ.get("PN_CPU_BUDGET_S", "420"))       # the sample does not depend on --steps / --warmup
    val, desc, cores, ms = cpu_baseline(budget)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": val, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc, "sample_seconds": ms},
            "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ CUDA path
def build_pipeline(device, seed):
    from panacea_b200.pipeline import DenoisingPipeline, default_sampler_config
    torch.manual_seed(seed)          # the default init draws on the device generator, which torch seeds at random per process
    with torch.device(device):
        pipe = DenoisingPipeline(sampler_config=default_sampler_config(50, 5.0), use_cuda_graph=True)
    pipe.model.randomize_zero_init(seed=seed)
    pipe.model.controlnet.randomize_zero_init(seed=seed + 1)
    return pipe


def synth_inputs_host(seed):
    """Synthetic conditioning + initial noise in PINNED host memory (what a data loader would hand over)."""
    g = torch.Generator().manual_seed(seed)
    Wt = VIEWS * W_VIEW
    hint = torch.rand(T, 19, 8 * H, 8 * Wt, generator=g)
    concat = torch.randn(T, 4, H, Wt, generator=g)
    c_txt = torch.randn(1, 77, 1024, generator=g)
    uc_txt = torch.randn(1, 77, 1024, generator=g)
    noise = torch.randn(T, 4, H, Wt, generator=g)
    pin = (lambda t: t.pin_memory()) if torch.cuda.is_available() else (lambda t: t)
    return {"hint": pin(hint), "concat": pin(concat), "c_txt": pin(c_txt), "uc_txt": pin(uc_txt), "noise": pin(noise)}


def load_traffic():
    """DRAM bytes per launch of the dominant kernel family from the committed ncu pass (tools/ncu_traffic.py)."""
    cands = sorted((ROOT / "profiles").glob("r*_gemm_traffic.json"))
    if not cands:
        return None, None
    try:
        d = json.loads(cands[-1].read_text())
        return d["dram_bytes_per_launch"], f"profiles/{cands[-1].name}: ncu dram__bytes_read.sum + dram__bytes_write.sum over the {d['launches']} gemm_tc launches of one eps-evaluation / launches"
    except (OSError, ValueError, KeyError):
        return None, None


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """Writes each device tensor as out_dir/<name>.npy in float32."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in arrays.items():
        np.save(d / f"{name}.npy", t.detach().float().cpu().numpy())
    log(f"wrote {', '.join(f'{n}.npy' for n in arrays)} to {d}")


def profile_dominant_kernel(pipe, x_in, t_dev, cc):
    """One eager eps-eval with CUDA-event timing around every launch of the dominant kernel (the tcgen05 GEMM /
    implicit-conv kernel): achieved TFLOP/s = sum of algorithmic FLOPs / sum of launch durations."""
    eng = pipe.model.engine()
    ops = eng.ops
    recs = []
    orig = ops.gemm

    def timed(a, w, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = orig(a, w, **kw)
        e.record()
        rows = a.numel() // a.shape[-1]
        n_out = w.shape[0] // 2 if kw.get("geglu") else w.shape[0]
        osz = 2 if kw.get("out_dtype", torch.float32) == torch.bfloat16 else 4
        abytes = 2.0 * rows * a.shape[-1] + 2.0 * w.numel() + osz * rows * n_out        # A + W + out (algorithmic, once each)
        for r in (kw.get("residual"), kw.get("residual2")):
            if r is not None:
                abytes += r.element_size() * rows * n_out
        recs.append((2.0 * rows * w.shape[0] * w.shape[1], s, e, abytes))
        return out

    # single-stream order for this pass: with the ControlNet and the UNet encoder on two streams (Engine.eps) a launch's
    # event pair would also span the time its CTAs queue behind the other branch's kernel
    two = eng.two_streams
    eng.two_streams = False
    eng.eps(x_in, cc["concat"].float().contiguous(), t_dev)      # untimed eager pass (module load, allocator warm-up)
    torch.cuda.synchronize()
    ops.gemm = timed
    try:
        eng.eps(x_in, cc["concat"].float().contiguous(), t_dev)
        torch.cuda.synchronize()
    finally:
        ops.gemm = orig
        eng.two_streams = two
    flops = sum(r[0] for r in recs)
    secs = sum(r[1].elapsed_time(r[2]) for r in recs) * 1e-3
    return flops, secs, len(recs), sum(r[3] for r in recs)


def run_ours(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from panacea_b200 import dist_utils as D
    seed = D.rank_seed(rank)                                       # inference.py:250: 3407 + rank
    log("building full-size UNet + ControlNet on the device")
    pipe = build_pipeline(dev, seed)
    log("synthetic host inputs (pinned)")
    host = synth_inputs_host(seed)
    ops = pipe.model.engine().ops                                  # packs bf16 operands
    log("weights packed")
    den, sampler, wrapper = pipe.denoiser, pipe.sampler, pipe.wrapper
    wrapper.hint_repeat = 2                                        # CFG halves share the BEV hint
    K, Wm = args.steps, args.warmup

    def upload():
        hint = host["hint"].to(dev, non_blocking=True)
        concat = host["concat"].to(dev, non_blocking=True)
        ctx = torch.cat([host["uc_txt"], host["c_txt"]]).to(dev, non_blocking=True)
        return {"cond_feat": hint, "concat": torch.cat([concat, concat]), "crossattn": ctx}

    cc = upload()
    sig = [float(s) for s in sampler.sigmas(50)]
    scal = [den.step_scalars(s) for s in sig[:-1]]
    n = T
    t_all = torch.tensor([[s[0]] * (2 * n) for s in scal], dtype=torch.int64, device=dev)
    x = ops.scale_dup(host["noise"].to(dev).float().contiguous(), math.sqrt(1.0 + sig[0] ** 2), 1)
    x_in = ops.scale_dup(x, scal[0][2], 2)

    def step(i):
        j = i % (len(sig) - 1)
        eps = wrapper(x_in, t_all[j], cc, return_static=True)
        ops.cfg_euler_step(x, eps, x_in, sig[j], sig[j + 1], 5.0, scal[j + 1][2] if j + 1 < len(scal) else scal[0][2], sigma_q=scal[j][1])
        return eps

    for i in range(max(Wm, 3)):                                    # >= 3 warm-ups: packing, graph capture, clocks
        step(i)
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    launches0 = ops.launches
    step(0)
    torch.cuda.synchronize()
    launches_per_replay = ops.launches - launches0                 # python-side launches outside the captured graph
    graph_launches = getattr(wrapper, "_graph_launches", None)

    # ---- timed region 1: device-resident (`value`)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(K):
        eps = step(i)
    ev1.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:                            # before the e2e region overwrites x and eps
        dump_outputs(args.dump_outputs, {"latent": x, "eps": eps})
    if dist is not None:
        dist.barrier()
    ms = ev0.elapsed_time(ev1)
    log(f"timed region: {K} steps in {ms:.1f} ms")
    clk = clocks.stop() if rank == 0 else None
    ms = D.max_over_ranks(ms, dev)

    # ---- timed region 2: end to end through the public API with host buffers (`e2e`)
    xh = torch.empty(n, 4, H, VIEWS * W_VIEW).pin_memory()
    xin_h = torch.empty(2 * n, 4, H, VIEWS * W_VIEW).pin_memory()
    xin_h.copy_(x_in.cpu())
    h2d = d2h = 0
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    wrapper.invalidate(drop_graph=False)                           # new sample, same shapes: the captured graph is reused
    cc2 = upload()                                                 # once per sample: conditioning H2D + hint stem + text K/V
    h2d += sum(host[k].numel() * 4 for k in ("hint", "concat", "c_txt", "uc_txt"))
    for i in range(K):
        j = i % (len(sig) - 1)
        xi = xin_h.to(dev, non_blocking=True)                      # this step's network input from pinned host memory
        ti = t_all[j]
        h2d += xin_h.numel() * 4
        eps = wrapper(xi, ti, cc2, return_static=True)
        ops.cfg_euler_step(x, eps, xi, sig[j], sig[j + 1], 5.0, scal[j + 1][2] if j + 1 < len(scal) else scal[0][2], sigma_q=scal[j][1])
        xh.copy_(x, non_blocking=True)                             # the step's result back to the host
        xin_h.copy_(xi, non_blocking=True)
        d2h += (xh.numel() + xin_h.numel()) * 4
        torch.cuda.current_stream().synchronize()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ms_e2e = e0.elapsed_time(e1)
    log(f"e2e region: {K} steps in {ms_e2e:.1f} ms")
    ms_e2e = D.max_over_ranks(ms_e2e, dev)
    # configs[2]: gather the final latents on rank 0 over NCCL (stand-in for decoded frames; the VAE is out of scope)
    gathered = D.gather_on_rank0(x)
    if rank == 0:
        log(f"gathered {len(gathered)} latent tensors of shape {tuple(x.shape)} on rank 0")

    # ---- dominant-kernel roofline (eager, per-launch CUDA events), launch count of one graphed eps-eval
    flops, secs, n_gemm, algo_bytes = profile_dominant_kernel(pipe, x_in, t_all[0], cc2)
    l0 = ops.launches
    pipe.model.engine().eps(x_in, cc2["concat"].float().contiguous(), t_all[0])
    torch.cuda.synchronize()
    launches_per_eps = ops.launches - l0
    log(f"profiled dominant kernel: {n_gemm} launches, {flops / secs / 1e12:.0f} TF/s; {launches_per_eps} launches per eps-eval")

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        log("CPU baseline (oracle port) ...")
        val, desc, cores, msc = cpu_baseline(float(os.environ.get("PN_CPU_BUDGET_S", "180")))    # same samples as --impl reference when they fit
        log(f"CPU baseline: {val:.5f} steps/s on {cores} cores")
        cpu = {"value": val, "unit": "steps/s", "cores": cores, "kind": "port", "sample": desc, "sample_seconds": msc}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except (OSError, ValueError):
            pass
        peak = peaks.get("bf16_tflops_sustained", 1400.0)
        achieved = flops / secs / 1e12
        traffic, traffic_src = load_traffic()
        value = world * K / (ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": K, "warmup": max(Wm, 3),
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "config": workload_config(world),
            "e2e": {"value": world * K / (ms_e2e * 1e-3), "unit": "steps/s", "h2d_bytes_per_step": h2d // K, "d2h_bytes_per_step": d2h // K,
                    "note": "per step: network input H2D from pinned memory + updated latent D2H; conditioning upload, BEV hint stem and "
                            "text K/V (once per sample) are inside the timed region"},
            "gpu_launches": (launches_per_eps + 1) * K,
            "launches_per_step": launches_per_eps + 1,
            "algorithmic_tflop_per_step": ALGO_TFLOP_PER_STEP,
            "achieved_tflops_whole_step": ALGO_TFLOP_PER_STEP * (K / (ms * 1e-3)),
            "roofline": {"bound": "tensor", "kernel": "pn::gemm_tc_kernel (tcgen05 GEMM / implicit conv, all launches of one eps-eval)",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                         "traffic_unit": "bytes per launch (DRAM read + write)", "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": algo_bytes / max(n_gemm, 1),
                         "algorithmic_flops_per_launch": flops / max(n_gemm, 1),
                         "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "fallback 1400",
                         "launches": n_gemm, "share_of_step": secs / (ms * 1e-3 / K),
                         "how": "sum of 2*M*N*K over the launches / sum of per-launch CUDA-event durations, eager pass after the timed region"},
            "clocks": clk, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's latent and eps as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — this implementation has no CPU path (use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: self-launch under torchrun when started as a plain script
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}", "--master-addr", "127.0.0.1",
               "--master-port", os.environ.get("MASTER_PORT", "29511"), str(Path(__file__).resolve()), "--gpus", str(args.gpus), "--steps",
               str(args.steps), "--warmup", str(args.warmup)] + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) \
            + (["--dump-outputs", str(Path(args.dump_outputs).resolve())] if args.dump_outputs else [])
        raise SystemExit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
