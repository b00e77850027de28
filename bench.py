#!/usr/bin/env python
"""bench.py -- mel-frames/s of the full reverse-diffusion loop (BASELINE.json metric).

One "step" = one complete pass of the hot path over one batch: the infer branch of GaussianDiffusion.forward after the
conditioner (start state, all sampler steps through DiffNet, denorm epilogue) for B utterances of T frames.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1|2|3|4|sweep] [--precision fp16s|fp16x2|fp16x3|fp16|fp32]
                  [--impl reference] [--dump-outputs DIR]

--config (BASELINE.json `configs`, default 2 = the configuration the metric is quoted on):
   1  DiffSpeech LJ   B=1  T=512   K=100  DDPM              (the reference's own CPU-runnable case)
   2  DiffSpeech      B=16 T=1024  K=100  DDPM              (headline)
   3  DiffSinger PopCS B=8 T=2048  K=1000 DDPM, beta <= 0.02, dilation cycle 4
   4  DiffSinger OpenCpop B=32 T=1024 PNDM (PLMS) interval 40 of K=1000 (25 steps, 26 evaluations), dilation cycle 4
   sweep  B in {1,4,16,64} x T in {256,1024,4096}, K in {25,100,1000} (K: 3 points at B=16,T=1024); one JSON line, points in "sweep"
Every line carries `roofline` (the residual-stack kernel against the measured sustained tensor peak), `cpu_baseline` (the
reference's PyTorch-CPU algorithm = oracle port on this box's host cores; plus `eager_cuda`: the same port on the GPU through
cuDNN / cuBLAS eager kernels, TF32 off and on) and `e2e` (through dsx_infer_host with pinned HOST buffers).

N > 1 (torchrun, one rank per GPU): utterance-sharded, B per GPU fixed (weak scaling), ONE all-gather of the finished mels
per step inside the timed region.  The strong-scaled BASELINE configs[3] (B=32 total, PLMS) is measured in the same run and
reported under extra.strong_config4.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

_JSON_OUT = sys.stdout
# algorithmic FLOPs per mel frame (SURVEY.md 8d): whole DiffNet evaluation, conditioner projection hoisted
FLOP_PER_FRAME_EVAL = 21184512
# the residual stack, per frame and layer: 2*(3*256*512 + 256*512)  (dilated conv + output projection, both halves)
FLOP_PER_FRAME_LAYER = 2 * (3 * 256 * 512 + 256 * 512)

CONFIGS = {
    "1": dict(B=1, T=512, K=100, sampler="ddpm", T_sched=100, max_beta=0.06, cycle=1,
              name="DiffSpeech LJSpeech B=1 T_frames=512 K=100 DDPM (BASELINE.json configs[0])"),
    "2": dict(B=16, T=1024, K=100, sampler="ddpm", T_sched=100, max_beta=0.06, cycle=1,
              name="DiffSpeech B=16 T_frames=1024 K=100 DDPM gaussian start, full reverse loop + denorm (BASELINE.json configs[1])"),
    "3": dict(B=8, T=2048, K=1000, sampler="ddpm", T_sched=1000, max_beta=0.02, cycle=4,
              name="DiffSinger PopCS B=8 T_frames=2048 full T=1000 DDPM (BASELINE.json configs[2])"),
    "4": dict(B=32, T=1024, K=1000, sampler="plms", interval=40, T_sched=1000, max_beta=0.02, cycle=4,
              name="DiffSinger OpenCpop B=32 T_frames=1024 PNDM (PLMS) interval 40 of K=1000 (BASELINE.json configs[3])"),
}
NOTES = {"fp16": "single MMA pass, fp16 round-to-nearest operands, tanh.approx gate: mel MAE 7e-5, max |d| 1.6e-3 after 100 steps (tests)",
         "fp16s": "single MMA pass, weights stochastically rounded into 64 sets cycled over the steps (unbiased, decorrelated weight "
                  "rounding), conditioner projection exact: max |d| 2.6e-4 after 100 steps (tests)",
         "fp16x2": "weights hi/lo split, 2 MMA passes, conditioner projection exact: max |d| 1.6e-4 after 100 steps (tests)",
         "fp16x3": "hi/lo split of both operands, 3 MMA passes: max |d| 1.4e-5 after 100 steps (tests)",
         "fp32": "CUDA-core fp32 path"}
DTYPES = {"fp16s": "f16 operands (weights stochastically rounded per step), 1 MMA pass, conditioner projection hoisted (f32), f32 accumulate and state",
          "fp16x2": "f16 operands, weights hi+lo split (2 MMA passes), conditioner projection hoisted (f32), f32 accumulate and state",
          "fp16x3": "f16 hi+lo split x3 MMA, f32 accumulate (fp32-equivalent)", "fp16": "f16 operands, f32 accumulate", "fp32": "f32"}
PASSES = {"fp16x3": 3.0, "fp16x2": 2.0, "fp16": 1.0, "fp16s": 1.0}


def hp_for(cfg):
    return dict(hidden_size=256, residual_layers=20, residual_channels=256, dilation_cycle_length=cfg["cycle"],
                audio_num_mel_bins=80, keep_bins=80)


def n_evals(cfg):
    if cfg["sampler"] == "plms":
        return len(range(0, cfg["K"], cfg["interval"])) + 1
    return cfg["K"]


def lj_spec_minmax():
    # value range of usr/configs/lj_ds_beta6.yaml (only its scale matters: it is a per-bin affine map)
    return torch.linspace(-4.6, -5.3, 80), torch.linspace(0.7, -0.2, 80)


def make_net(dsx, cfg, dev=None):
    torch.manual_seed(0)
    net = dsx.DiffNet(80, hparams=hp_for(cfg))
    torch.nn.init.normal_(net.output_projection.weight, std=0.02)
    return net.eval() if dev is None else net.to(dev).eval()


def make_inputs(B, T, rank):
    g = torch.Generator().manual_seed(1234 + 7919 * rank)
    cond = torch.randn(B, T, 256, generator=g)            # frames-major, handed over as the transposed view
    g2 = torch.Generator().manual_seed(1235 + 7919 * rank)
    xT = torch.randn(B, 1, 80, T, generator=g2)
    return cond, xT


def schedule_for(cfg):
    """The 12 registered buffers (shallow_diffusion_tts.py:90-123) through the package's own mirror (no oracle import
    on the product arm)."""
    from diffsinger_b200.modules import linear_beta_schedule, register_schedule_buffers
    from diffsinger_b200 import _capi

    class Holder(torch.nn.Module):
        pass

    m = Holder()
    register_schedule_buffers(m, linear_beta_schedule(cfg["T_sched"], cfg["max_beta"]), [0.0] * 80, [1.0] * 80, 80)
    return {n: getattr(m, n) for n in _capi.SCHEDULE_BUFFERS}


class ClockSampler:
    """SM clock / throttle reasons / board power DURING the timed region: an NVML polling thread (5 ms period; the NVML
    calls release the GIL and the timed loop only enqueues launches and waits), every sample time-stamped so that only
    those between mark_start() and mark_end() count.  Falls back to an `nvidia-smi -lms` subprocess (the recipe's clocks
    line) when NVML cannot be loaded."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        import threading
        self.samples, self.t0, self.t1, self.mx = [], None, None, None
        self.stop = threading.Event()
        self.thread, self.proc = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(v.strip().isdigit() for v in vis.split(",")) else index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None
            self.path = f"/tmp/dsx_clocks_{os.getpid()}_{index}.csv"
            try:
                self.f = open(self.path, "w")
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                              "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                             stderr=subprocess.DEVNULL)
            except Exception:
                self.proc = None

    def _poll(self):
        nv, h = self.nv, self.h
        reasons_fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop.is_set():
            try:
                clk = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                bits = int(reasons_fn(h))
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    watts = None
                self.samples.append((time.time(), clk, bits, watts))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.thread is None:
            time.sleep(0.3)          # let the first nvidia-smi samples land
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def finish(self):
        if self.t1 is None:
            self.t1 = time.time()
        if self.thread is not None:
            self.stop.set()
            self.thread.join(timeout=2)
            inside = [x for x in self.samples if self.t0 <= x[0] <= self.t1] or self.samples
            if not inside:
                return {"sm_mhz": None, "sm_max_mhz": self.mx, "reasons": [], "samples": 0}
            bits = 0
            for x in inside:
                bits |= x[2]
            watts = [x[3] for x in inside if x[3] is not None]
            return {"sm_mhz": float(np.median([x[1] for x in inside])), "sm_min_mhz": float(min(x[1] for x in inside)),
                    "sm_max_mhz": self.mx, "reasons": sorted(n for b, n in self.BITS.items() if bits & b),
                    "samples": len(inside), "power_w": float(np.median(watts)) if watts else None,
                    "how": "NVML, 5 ms period, samples inside the timed region only"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=3)
        except Exception:
            self.proc.kill()
        self.f.close()
        clk, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 6:
                continue
            try:
                clk.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        try:
            os.remove(self.path)
        except OSError:
            pass
        # samples under load only (idle samples sit at the floor clock)
        load = [c for c in clk if c > 0.5 * (mx or 1)] or clk
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(clk), "how": "nvidia-smi -lms 100"}


# ------------------------------------------------------------------------------------------------------------------
# baselines: the reference's algorithm (oracle port = the ATen kernels the reference itself runs) on the host cores and,
# for context, eagerly on the GPU.  These legs are the only users of oracle/ in this file.
# ------------------------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """MKL-DNN does not always scale to every core of a big host: time a tiny p_sample at a few thread counts
    and keep the fastest (so the CPU baseline is the best the host can do, not an oversubscribed one)."""
    from oracle import diffnet_oracle as O
    n = os.cpu_count() or 1
    cands = sorted({n, min(n, 64), min(n, 32), min(n, 16)}, reverse=True)
    sd = O.build_state_dict(0)
    S = O.make_schedule(O.linear_beta_schedule(100, 0.06))
    cond, x = make_inputs(4, 256, 0)
    cond = cond.transpose(1, 2)
    best = (None, 1e30)
    for c in cands:
        torch.set_num_threads(c)
        with torch.no_grad():
            O.p_sample(sd, S, x, 50, cond, x)
            t0 = time.perf_counter()
            for _ in range(2):
                O.p_sample(sd, S, x, 50, cond, x)
            dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (c, dt)
    return best[0]


def cpu_baseline(cfg, n_steps, threads=None, budget_s=30.0):
    """Seconds per DiffNet evaluation + sampler update of the reference's CPU path at this config's (B, T): the median of
    `n_steps` (>= 3) consecutive p_sample steps (their cost does not depend on t), stopping early at `budget_s`."""
    from oracle import diffnet_oracle as O
    cores = threads or pick_cpu_threads()
    torch.set_num_threads(cores)
    sd = O.build_state_dict(0, dilation_cycle_length=cfg["cycle"])
    S = O.make_schedule(O.linear_beta_schedule(cfg["T_sched"], cfg["max_beta"]))
    cond, x = make_inputs(cfg["B"], cfg["T"], 0)
    cond = cond.transpose(1, 2)
    g = torch.Generator().manual_seed(1236)
    per = []
    with torch.no_grad():
        noise = torch.randn(x.shape, generator=g)
        t_hi = cfg["T_sched"] - 1
        x = O.p_sample(sd, S, x, t_hi, cond, noise, cfg["cycle"])          # warm-up (thread pool, allocator)
        t_begin = time.perf_counter()
        for j in range(n_steps):
            t0 = time.perf_counter()
            x = O.p_sample(sd, S, x, t_hi - 1 - j, cond, noise, cfg["cycle"])
            per.append(time.perf_counter() - t0)
            if time.perf_counter() - t_begin > budget_s and len(per) >= 3:
                break
    return float(np.median(per)), cores, len(per)


def eager_cuda_baseline(cfg, dev, n_steps=3):
    """The same port with its tensors on the GPU: PyTorch-eager cuDNN / cuBLAS kernels (what the reference runs with
    `.cuda()`), TF32 off and on.  Seconds per evaluation + update, CUDA events."""
    from oracle import diffnet_oracle as O
    sd = {k: v.to(dev) for k, v in O.build_state_dict(0, dilation_cycle_length=cfg["cycle"]).items()}
    S = {k: v.to(dev) for k, v in O.make_schedule(O.linear_beta_schedule(cfg["T_sched"], cfg["max_beta"])).items()}
    cond, x = make_inputs(cfg["B"], cfg["T"], 0)
    cond, x = cond.to(dev).transpose(1, 2), x.to(dev)
    noise = torch.randn_like(x)
    out = {}
    orig_arange, orig_full = torch.arange, torch.full
    # the port creates its index / frequency tensors on the default device
    torch.set_default_device(dev)
    try:
        for name, tf32 in (("tf32_off", False), ("tf32_on", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            t_hi = cfg["T_sched"] - 1
            with torch.no_grad():
                xx = x
                for j in range(2):
                    xx = O.p_sample(sd, S, xx, t_hi - j, cond, noise, cfg["cycle"])
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for j in range(n_steps):
                    xx = O.p_sample(sd, S, xx, t_hi - 2 - j, cond, noise, cfg["cycle"])
                e1.record()
                torch.cuda.synchronize()
            out[name] = e0.elapsed_time(e1) * 1e-3 / n_steps
    finally:
        torch.set_default_device("cpu")
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = True
    return out


def run_reference_arm(args, cfg, rank, world):
    """`--impl reference`: the reference's own CPU path (oracle port, pinned bit-exact to the live reference by
    oracle/gen_golden.py) timed on the host cores, on this arm's config / metric / unit."""
    if rank != 0:
        return
    B, T = cfg["B"], cfg["T"]
    evals = n_evals(cfg)
    threads = pick_cpu_threads()
    per = []
    for i in range(min(args.warmup, 1) + args.steps):
        dt, cores, n = cpu_baseline(cfg, max(3, args.ref_evals), threads, budget_s=40.0)
        if i >= min(args.warmup, 1):
            per.append(dt)
    step_s = float(np.mean(per)) * evals
    value = B * T / step_s
    line = {
        "impl": "reference", "metric": "mel-frames/s", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["name"], "B_per_gpu": B, "T_frames": T, "K": cfg["K"], "layers": 20, "channels": 256,
                   "evaluations_per_step": evals},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"median of {n} consecutive p_sample steps at B={B},T={T} per bench step, x{evals} evaluations "
                                   "extrapolated (per-step cost is independent of t)"},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_JSON_OUT, flush=True)


# ------------------------------------------------------------------------------------------------------------------
class Arm:
    """One sampler + inputs for a config on this rank."""

    def __init__(self, dsx, cfg, prec, dev, rank, B=None):
        from diffsinger_b200 import _capi
        self.cfg, self.dev, self.capi = cfg, dev, _capi
        self.B = cfg["B"] if B is None else B
        self.T = cfg["T"]
        self.net = make_net(dsx, cfg, dev)
        self.s = dsx.DsxSampler(self.net, prec, cfg["cycle"])
        self.s.ensure_weights(dev)
        self.s.set_schedule(schedule_for(cfg))
        smin, smax = lj_spec_minmax()
        self.smin_h, self.smax_h = smin, smax
        self.smin, self.smax = smin.to(dev), smax.to(dev)
        self.cond_h, self.xT_h = make_inputs(self.B, self.T, rank)
        self.cond = self.cond_h.to(dev).transpose(1, 2)
        self.xT = self.xT_h.to(dev)
        self.interval = cfg.get("interval", 0) if cfg["sampler"] == "plms" else 0

    def step(self, i):
        return self.s.infer(self.cond, self.cfg["K"], self.smin, self.smax, x_start=self.xT, seed=1236 + i,
                            pndm_interval=self.interval)

    def close(self):
        self.s.close()


def timed_steps(arm, steps, warmup, world, dev, flush, gather_total=None, clocks_index=None):
    from diffsinger_b200.parallel import all_gather_batch

    def step(i):
        mel = arm.step(i)
        if world > 1 and gather_total:
            mel = all_gather_batch(mel, gather_total)
        return mel

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    cs = ClockSampler(clocks_index) if clocks_index is not None else None
    if cs:
        cs.start()
    l0 = arm.s.info(arm.capi.INFO_KERNEL_LAUNCHES)
    times = []
    for i in range(steps):
        flush.zero_()                                          # L2 flush between timed iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        mel = step(warmup + i)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    l1 = arm.s.info(arm.capi.INFO_KERNEL_LAUNCHES)
    if cs:
        cs.mark_end()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    clk = cs.finish() if cs else None
    total_ms = torch.tensor([sum(times)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    assert torch.isfinite(mel).all()
    return float(total_ms.item()), (l1 - l0), clk, mel


def roofline_of(arm, prec, ms_per_step):
    """The dominant kernel, CUDA events around its launches on the launching stream (DSX_OPT_PROFILE).  With the fused head
    (default) that kernel is the whole diffusion step -- residual stack, skip GEMM, head projections, sampler update, next
    input projection -- so its algorithmic FLOPs are those of a whole DiffNet evaluation; `stack_only` repeats the
    measurement with the head as a separate kernel (DSX_OPT_FUSED_HEAD = 0): the residual stack alone, the quantity round 1
    reported."""
    capi = arm.capi
    cfg, B, T = arm.cfg, arm.B, arm.T
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("bf16_tflops_sustained", 1400.0)

    def profile(fused):
        arm.s.set_option(capi.OPT_FUSED_HEAD, 1 if fused else 0)
        arm.step(98)
        arm.s.set_option(capi.OPT_PROFILE, 1)
        arm.step(99)
        ns, n = arm.s.info(capi.INFO_LAYER_KERNEL_NS), arm.s.info(capi.INFO_LAYER_KERNEL_LAUNCHES)
        arm.s.set_option(capi.OPT_PROFILE, 0)
        return ns, n, ns * 1e-9 / max(n, 1)       # brackets are per evaluation (every launch group)

    ns_s, n_s, t_stack = profile(False)
    ns, n, t_eval = profile(True)
    stack_launches = arm.s.info(capi.INFO_STACK_KERNEL_LAUNCHES)
    traffic, traffic_note = None, "not captured for this configuration"
    try:     # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this kernel, per launch
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_stack_traffic.json")))
        if cfg is CONFIGS["2"] and prec in tj:
            traffic = tj[prec]["dram_bytes_read"] + tj[prec]["dram_bytes_write"]
            traffic_note = tj.get("note", "static: from the committed ncu capture of this command (profiles/), not re-measured by this run")
    except Exception:
        pass
    flops_stack = FLOP_PER_FRAME_LAYER * B * T * 20
    flops_eval = FLOP_PER_FRAME_EVAL * B * T
    fused = bool(stack_launches) and arm.s.info(capi.INFO_KERNEL_LAUNCHES) > 0
    kernel = ("k_tc_stack (dsx_stack.cu, tcgen05): the whole diffusion step in one launch -- residual stack with x in registers / y in shared "
              "memory, deferred skip GEMM, head projections, sampler update, next input projection") if stack_launches else \
        "k_tc_layer (dsx_tc.cu: round-1 residual-stack kernel)"
    ach = flops_eval / t_eval / 1e12
    whole = FLOP_PER_FRAME_EVAL * B * T * n_evals(cfg) / (ms_per_step * 1e-3) / 1e12
    return {"bound": "tensor", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
            "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
            "traffic": traffic, "traffic_note": traffic_note,
            "flops_per_launch": flops_eval, "avg_launch_us": t_eval * 1e6, "evaluations_profiled": n,
            "kernel_share_of_step": ns * 1e-6 / ms_per_step, "mma_passes": PASSES.get(prec),
            "stack_only": {"note": "head as a separate kernel (DSX_OPT_FUSED_HEAD = 0): the 20 residual layers + skip GEMM alone",
                           "achieved": flops_stack / t_stack / 1e12, "frac": flops_stack / t_stack / 1e12 / peak,
                           "flops_per_launch": flops_stack, "avg_launch_us": t_stack * 1e6, "avg_layer_us": t_stack * 1e6 / 20,
                           "evaluations_profiled": n_s},
            "whole_step_algorithmic_tflops": whole, "whole_step_frac": whole / peak}


def e2e_of(dsx, cfg, prec, dev, rank, world, steps):
    """Same metric through the C ABI with HOST buffers (H2D of cond + x_T, D2H of mel inside the timed region)."""
    arm = Arm(dsx, cfg, prec, dev, rank)
    B, T = arm.B, arm.T
    cond_p, xT_p = arm.cond_h.pin_memory(), arm.xT_h.pin_memory()
    out_p = torch.empty(B, T, 80).pin_memory()
    cond_view = cond_p.transpose(1, 2)
    kw = dict(x_start=xT_p, out=out_p, device=dev, pndm_interval=arm.interval)
    for i in range(2):
        arm.s.infer_host(cond_view, cfg["K"], arm.smin_h, arm.smax_h, seed=5 + i, **kw)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        arm.s.infer_host(cond_view, cfg["K"], arm.smin_h, arm.smax_h, seed=50 + i, **kw)
    torch.cuda.synchronize()
    e2e_s = torch.tensor([(time.perf_counter() - t0) / steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    arm.close()
    return {"value": world * B * T / float(e2e_s.item()), "unit": "frames/s",
            "h2d_bytes_per_step": int(cond_p.numel() * 4 + xT_p.numel() * 4 + 2 * 80 * 4),
            "d2h_bytes_per_step": int(out_p.numel() * 4), "ms_per_step": float(e2e_s.item()) * 1e3,
            "api": "dsx_infer_host (C ABI, pinned host buffers)"}


def bench_config(dsx, cfg, prec, args, dev, rank, world, local_rank, flush, full=True, keep_output=False):
    arm = Arm(dsx, cfg, prec, dev, rank)
    B, T = arm.B, arm.T
    total_ms, launches, clk, mel = timed_steps(arm, args.steps, args.warmup, world, dev, flush, gather_total=B * world,
                                               clocks_index=local_rank)
    ms = total_ms / args.steps
    out = {"value": world * B * T / (ms * 1e-3), "ms_per_step": ms, "launches": int(launches), "clocks": clk,
           "mel": mel.cpu() if keep_output else None,
           "roofline": roofline_of(arm, prec, ms) if prec != "fp32" else None,
           "workspace_bytes": arm.s.info(arm.capi.INFO_WORKSPACE_BYTES)}
    arm.close()
    if full:
        out["e2e"] = e2e_of(dsx, cfg, prec, dev, rank, world, max(2, min(args.steps, 3)))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dsx", choices=["dsx", "reference"])
    ap.add_argument("--config", default="2", choices=["1", "2", "3", "4", "sweep"])
    ap.add_argument("--precision", default=os.environ.get("DSX_BENCH_PRECISION", "fp16s"))
    ap.add_argument("--ref-evals", type=int, default=3)
    ap.add_argument("--cpu-evals", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the mel of the last timed step (what the caller receives, [B, T, 80]) as DIR/mel.npy, float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the dsx arm; the reference arm only times the CPU path")

    # stdout carries exactly ONE JSON line: everything libraries print there (NCCL's version banner, ...) goes to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = CONFIGS["2" if args.config == "sweep" else args.config]
    if args.impl == "reference":
        run_reference_arm(args, cfg, rank, world)
        return

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__
    __graft_entry__.build()
    import diffsinger_b200 as dsx

    prec = args.precision
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)       # > 126 MB L2
    main_res = bench_config(dsx, cfg, prec, args, dev, rank, world, local_rank, flush, keep_output=bool(args.dump_outputs))
    B, T, K = cfg["B"], cfg["T"], cfg["K"]
    if args.dump_outputs and rank == 0:
        # inputs, weights and noise seeds depend on the arguments alone, so two builds run with the same arguments can be
        # compared output for output
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "mel.npy"), main_res.pop("mel").numpy().astype(np.float32))

    extra = {}
    if not args.no_extra and world == 1 and args.config != "sweep":
        for other in ("fp16x3", "fp16x2", "fp16s", "fp16"):
            if other == prec:
                continue
            arm = Arm(dsx, cfg, other, dev, rank)
            tms, _, _, _ = timed_steps(arm, 2, 2, world, dev, flush)
            arm.close()
            extra[other] = {"value": B * T / (tms / 2 * 1e-3), "unit": "frames/s", "ms_per_step": tms / 2, "note": NOTES[other]}
    if not args.no_extra and world > 1 and 32 % world == 0:
        # BASELINE configs[3] strong-scaled: B = 32 utterances in total, 32 / N per GPU, one all-gather per step
        c4 = CONFIGS["4"]
        arm = Arm(dsx, c4, prec, dev, rank, B=32 // world)
        tms, _, _, _ = timed_steps(arm, 2, 2, world, dev, flush, gather_total=32)
        arm.close()
        extra["strong_config4"] = {"value": 32 * c4["T"] / (tms / 2 * 1e-3), "unit": "frames/s", "ms_per_step": tms / 2, "scaling": "strong",
                                   "workload": c4["name"], "B_total": 32, "B_per_gpu": 32 // world,
                                   "note": "compare with --config 4 at --gpus 1 (same total work)"}

    sweep = None
    if args.config == "sweep" and world == 1:
        sweep = []
        quick = argparse.Namespace(steps=1, warmup=1)
        for Bs in (1, 4, 16, 64):
            for Ts in (256, 1024, 4096):
                c = dict(CONFIGS["2"], B=Bs, T=Ts, K=25, name=f"sweep B={Bs} T={Ts} K=25")
                r = bench_config(dsx, c, prec, quick, dev, rank, world, local_rank, flush, full=False)
                sweep.append({"B": Bs, "T": Ts, "K": 25, "frames_per_s": r["value"], "ms_per_step": r["ms_per_step"],
                              "roofline_frac": r["roofline"]["frac"] if r["roofline"] else None,
                              "stack_only_frac": r["roofline"]["stack_only"]["frac"] if r["roofline"] else None,
                              "workspace_bytes": r["workspace_bytes"]})
        for Ks, Tsch, mb in ((25, 100, 0.06), (100, 100, 0.06), (1000, 1000, 0.02)):
            c = dict(CONFIGS["2"], K=Ks, T_sched=Tsch, max_beta=mb, name=f"sweep B=16 T=1024 K={Ks}")
            r = bench_config(dsx, c, prec, quick, dev, rank, world, local_rank, flush, full=False)
            sweep.append({"B": 16, "T": 1024, "K": Ks, "frames_per_s": r["value"], "ms_per_step": r["ms_per_step"],
                          "roofline_frac": r["roofline"]["frac"] if r["roofline"] else None})

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        dt, cores, n = cpu_baseline(cfg, args.cpu_evals)
        evals = n_evals(cfg)
        cpu = {"value": B * T / (dt * evals), "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": f"median of {n} consecutive p_sample steps at B={B},T={T} (oracle port of the reference's PyTorch-CPU path), "
                         f"x{evals} evaluations extrapolated", "ms_per_diffnet_step": dt * 1e3}
        try:
            eg = eager_cuda_baseline(cfg, dev)
            cpu["eager_cuda"] = {k: {"value": B * T / (v * evals), "unit": "frames/s", "ms_per_diffnet_step": v * 1e3}
                                 for k, v in eg.items()}
            cpu["eager_cuda"]["note"] = ("the same port with its tensors on this GPU (PyTorch eager: cuDNN convs / cuBLAS, ~300 ATen "
                                         "launches per step); context only, not the reference arm")
        except Exception as e:  # noqa: BLE001
            cpu["eager_cuda"] = {"error": str(e)[:200]}

    if rank == 0:
        line = {
            "metric": "mel-frames/s", "value": main_res["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPES[prec], "data": "synthetic",
            "config": {"workload": cfg["name"], "B_per_gpu": B, "T_frames": T, "K": K, "layers": 20, "channels": 256,
                       "evaluations_per_step": n_evals(cfg), "precision": prec, "precision_note": NOTES[prec],
                       "noise": "in-kernel Philox4x32-10", "l2": "256 MB buffer written between timed iterations (L2 flush)",
                       "parallelism": f"utterance-sharded x{world}, one all-gather per step" if world > 1 else "single GPU"},
            "diffnet_step_ms": main_res["ms_per_step"] / n_evals(cfg),
            "roofline": main_res["roofline"], "cpu_baseline": cpu, "e2e": main_res.get("e2e"),
            "gpu_launches": main_res["launches"], "clocks": main_res["clocks"], "extra": extra,
        }
        if sweep is not None:
            line["sweep"] = sweep
        print(json.dumps(line), file=_JSON_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
