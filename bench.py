#!/usr/bin/env python
"""bench.py -- images/sec of the ViT forward hot path on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload vit_b16|vit_l16_map|clip_b32|siglip_b16|siglip2_l16_512]
                    [--dump-outputs DIR]

A "step" is one forward pass of the hot path over one synthetic batch; every timed loop below runs K steps.  Inputs and weights
come from fixed seeds, so the same arguments give the same inputs on every run, and `--dump-outputs DIR` writes what the last timed
step of the headline loop returned (see dump_outputs) so that two builds can be compared output for output.
The default workload is BASELINE.json configs[1]:
ViT-B/16 @224, batch 256 per GPU, fp16 tensor-core operands (fp32 accumulate / residual / LN / softmax), random-init weights.
  value  : whole-job images/sec with the inputs already resident in HBM (CUDA events, barrier + synchronize both sides,
           max over ranks).  Weak scaling: every rank runs its own 256-image batch; no data-path collective for ViT.
  e2e    : the same metric through the public Python API with HOST (pinned) inputs: H2D copy + forward + D2H of the logits
           inside the timed region (jimm_vit_forward_host), with a synchronisation every step.  `pipelined_depth2_value` is the
           same loop through `forward_async` with two calls in flight (every step still copies its inputs in and its result out);
           it is an extra, not the headline.
  roofline: the dominant kernel (tcgen05 GEMM) timed live with CUDA events around every launch of the timed steps.
  cpu_baseline: the CPU oracle (torch fp32, jimm semantics -- the stand-in for the reference's JAX-CPU path, which cannot
           be installed here) on a bounded sample, rank 0 / N=1 only.
  extra_workloads (N=1): north_star's second headline (SigLIP-B/16 @256) and BASELINE configs[2] (ViT-L/16 @384 MAP, bf16), K steps
           each: value, e2e and the live GEMM roofline, so that one run measures them too.
  collective (N>1): after the ViT leg every rank runs the dual-tower path the batch-sharded reference resolves with an all-gather
           (models/clip.py:183-187 under P("batch") inputs, examples/clip_inference.py:41-44): CLIP-B/32 at N<=4 (BASELINE configs[3] at N=4),
           SigLIP2-L/16 @512 at N=8 (configs[4]).  Reports pairs/s (device and e2e), the fused normalise + NVLink peer-store + logits kernel
           timed alone with CUDA events, bytes per peer, achieved NVLink GB/s against the measured 770 GB/s, and whether the sharded
           logits are bit-identical to the single-GPU head on the gathered embeddings (checked outside the timed region).
--impl reference times that CPU path alone, on the same metric / config (see the tier's reference-arm contract).
"""

from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GFLOP_PER_IMG = {"vit_b16": 35.128, "vit_l16_map": 383.85, "clip_b32": 14.778, "siglip_b16": 57.85, "siglip2_l16_512": 766.55}  # SURVEY.md 8(d)

WORKLOADS = {
    # name: (description, per-GPU batch, dtype)
    "vit_b16": ("ViT-B/16 @224, batch 256/GPU, fp16 operands, random-init (BASELINE configs[1])", 256, "float16"),
    "vit_l16_map": ("ViT-L/16 @384 MAP head, batch 128/GPU, bf16 operands (BASELINE configs[2])", 128, "bfloat16"),
    "clip_b32": ("CLIP ViT-B/32 dual tower, batch 256 pairs/GPU, fp16 (BASELINE configs[3])", 256, "float16"),
    "siglip_b16": ("SigLIP-B/16 @256 dual tower, batch 256 pairs/GPU, fp16 (north-star extra)", 256, "float16"),
    "siglip2_l16_512": ("SigLIP2-L/16 @512 dual tower (S=1024), batch 256 pairs/GPU, bf16, vocab 32000 stand-in (BASELINE configs[4] per-GPU share)",
                        256, "bfloat16"),
}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1402.5), d.get("hbm_gbs", 6568.4), "measured (MEASURED_PEAKS.json, sustained bf16 GEMM)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md 'clocks line')."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []   # (arrival time, csv line)
        self.proc = None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def in_window(self) -> int:
        """Samples that arrived while the timed region ran (a sample describes the ~100 ms before it arrives)."""
        if self.t0 is None or self.t1 is None:
            return len(self.rows)
        return sum(1 for t, _ in self.rows if self.t0 <= t <= self.t1 + 0.12)

    def selected_rows(self):
        """Samples of the timed region; if the region was too short for one, those of the post-region load the caller kept running
        (single GPU) or, failing that, the last warm-up samples (multi-GPU runs cannot extend the load unilaterally)."""
        if self.t0 is None or self.t1 is None:
            return list(self.rows)
        lo = self.t0 if self.in_window() else self.t1
        return [(t, r) for t, r in self.rows if t >= lo] or self.rows[-3:]

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for _, r in self.selected_rows():
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
def synthetic_tokens(B: int, T: int, V: int, kind: str, seed: int):
    """SURVEY.md 8(d): ids uniform in [1, V-2]; CLIP rows get one EOT = V-1 at a random position >= 1 (argmax pooling, models/clip.py:164);
    SigLIP rows are full length (last-token pooling, models/siglip.py:151)."""
    import torch

    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(1, V - 1, (B, T), generator=g, dtype=torch.int64)
    if kind == "clip":
        pos = torch.randint(1, T, (B,), generator=g)
        ids[torch.arange(B), pos] = V - 1
    return ids


def build_model(workload: str, dtype_name: str):
    """Random-init weights of the named architecture (no network for checkpoints): the reference's init distributions."""
    import torch

    from jimm_b200 import Rngs
    from jimm_b200.common.vit import VisionTransformerBase
    from jimm_b200.models import CLIP, SigLIP, VisionTransformer

    dt = getattr(torch, dtype_name)
    if workload == "vit_b16":
        return VisionTransformer(dtype=dt, rngs=Rngs(0)).eval(), 224, None
    if workload == "vit_l16_map":
        return VisionTransformerBase(img_size=384, patch_size=16, in_channels=3, hidden_size=1024, num_layers=24, num_heads=16, mlp_dim=4096,
                                     pooling_type="MAP", layernorm_epsilon=1e-6, dtype=dt, rngs=Rngs(0)), 384, None
    if workload == "clip_b32":
        return CLIP(224, 12, 768, 32, 77, 49408, 512, 8, 12, dtype=dt, rngs=Rngs(0)), 224, (77, 49408, "clip")
    if workload == "siglip_b16":
        return SigLIP(256, 12, 768, 16, 64, 32000, 768, 12, 12, dtype=dt, rngs=Rngs(0)), 256, (64, 32000, "siglip")
    if workload == "siglip2_l16_512":
        # vision 1024/24L/16H patch 16 @512 (S = 1024, MAP head), text 1024/24L/16H/T64 (SURVEY.md 8 table); the embedding gather
        # does not depend on the vocabulary size, 32000 keeps the random init short
        return SigLIP(512, 24, 1024, 16, 64, 32000, 1024, 16, 24, dtype=dt, rngs=Rngs(0)), 512, (64, 32000, "siglip")
    raise SystemExit(f"unknown workload {workload}")


def cpu_threads() -> int:
    """Threads for the CPU arm: every core this process may use (affinity mask and cgroup CPU quota honoured); JIMM_CPU_THREADS overrides."""
    env = os.environ.get("JIMM_CPU_THREADS")
    if env:
        return max(1, int(env))
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def oracle_step_fn(workload: str, B: int):
    """The CPU arm: oracle restatement in torch fp32 with jimm semantics, same architecture / synthetic inputs."""
    import torch

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import jimm_oracle as O

    torch.set_num_threads(cpu_threads())
    if workload == "vit_b16":
        cfg = O.ViTCfg()
        p = O.random_vit_params(cfg, seed=0)
        img = O.synthetic_images(B, 224)
        return lambda: O.vit_forward(p, cfg, img)
    if workload == "vit_l16_map":
        t = O.TowerCfg(384, 16, 3, 1024, 24, 16, 4096, "MAP", layernorm_epsilon=1e-6)
        p = O.random_tower_params(t, seed=0)
        img = O.synthetic_images(B, 384)
        return lambda: O.vision_tower(p, "", img, t)
    if workload == "clip_b32":
        cfg = O.DualCfg(224, 12, 768, 32, 77, 49408, 512, 8, 12)
        p = O.random_dual_params(cfg, "clip", seed=0)
        img, txt = O.synthetic_images(B, 224), O.synthetic_tokens(B, 77, 49408, "clip")
        return lambda: O.clip_forward(p, cfg, img, txt)
    if workload == "siglip2_l16_512":
        cfg = O.DualCfg(512, 24, 1024, 16, 64, 32000, 1024, 16, 24)
        p = O.random_dual_params(cfg, "siglip", seed=0)
        img, txt = O.synthetic_images(B, 512), O.synthetic_tokens(B, 64, 32000, "siglip")
        return lambda: O.siglip_forward(p, cfg, img, txt)
    cfg = O.DualCfg(256, 12, 768, 16, 64, 32000, 768, 12, 12)
    p = O.random_dual_params(cfg, "siglip", seed=0)
    img, txt = O.synthetic_images(B, 256), O.synthetic_tokens(B, 64, 32000, "siglip")
    return lambda: O.siglip_forward(p, cfg, img, txt)


def time_cpu(workload: str, B: int, steps: int, warmup: int):
    import torch

    fn = oracle_step_fn(workload, B)
    with torch.no_grad():
        for _ in range(warmup):
            fn()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        dt = time.perf_counter() - t0
    return B * steps / dt, dt / steps * 1e3


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference arm: the CPU restatement of the reference's forward (oracle/jimm_oracle.py, torch fp32, jimm semantics;
    the reference's own JAX-CPU path cannot be installed in this image) on the host cores, same metric / config."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # bounded sample: size the per-step batch from one probe image so a step stays around 3 s of host time
    probe_ips, _ = time_cpu(args.workload, 1, 1, 1)
    B = args.cpu_batch if args.cpu_batch_fixed else max(1, min(16, int(probe_ips * 3.0)))
    ips, ms = time_cpu(args.workload, B, args.steps, args.warmup)
    cores = cpu_threads()
    sample = f"{B} images/step x {args.steps} steps of {WORKLOADS[args.workload][0]}"
    line = {
        "impl": "reference", "metric": "images/sec", "value": ips, "unit": "images/sec", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOADS[args.workload][0], "cpu_sample_batch": B},
        "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": cores, "host_cores": os.cpu_count() or 1, "kind": "port", "sample": sample,
                         "note": "oracle/jimm_oracle.py (torch CPU fp32, jimm semantics); the reference's JAX-CPU path is not installable here"},
        "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0


DUMP_BYTES = 64 << 20


def dump_outputs(directory: str, arrays: dict, rank: int, world: int) -> list:
    """Write each {name: tensor} as `directory/<name>.npy` (`<name>.rank<r>.npy` when world > 1) in float32.  The files of all ranks
    stay within DUMP_BYTES: an array over its share is replaced by a fixed sample of its flattened elements (the same indices on
    every run, in ascending order), so that dumps of two builds still line up element for element."""
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    budget = DUMP_BYTES // (world * len(arrays))
    written = []
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.nbytes > budget:
            idx = np.sort(np.random.default_rng(0).choice(a.size, budget // a.itemsize, replace=False))
            a = a.reshape(-1)[idx]
        path = os.path.join(directory, f"{name}.npy" if world == 1 else f"{name}.rank{rank}.npy")
        np.save(path, a)
        written.append(path)
    return written


def gemm_roofline(lib, native, step_dev, steps, ms_step):
    """The dominant kernel (tcgen05 GEMM) timed live: CUDA events on the launch stream around every launch of `steps` steps."""
    from jimm_b200 import _lib

    _lib.check(lib.jimm_profile_begin(native.handle))
    for _ in range(steps):
        step_dev()
    g_ms, g_fl, g_n = C.c_double(), C.c_double(), C.c_longlong()
    _lib.check(lib.jimm_profile_end(native.handle, C.byref(g_ms), C.byref(g_fl), C.byref(g_n)))
    peak_tf, _, peak_src = peaks()
    achieved = g_fl.value / (g_ms.value * 1e-3) / 1e12 if g_ms.value > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    return {"bound": "tensor", "kernel": "gemm_tcgen05_kernel", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
            "frac": achieved / peak_tf, "traffic": traffic, "peak_source": peak_src, "launches": g_n.value,
            "avg_launch_ms": g_ms.value / max(g_n.value, 1), "gemm_share_of_step": g_ms.value / steps / ms_step}


class Bench:
    """One workload on this rank's GPU: model, synthetic inputs (device-resident, pinned fp32 host, pinned uint8 host) and timers."""

    def __init__(self, workload, batch, rank, world, local, lib):
        import torch

        from jimm_b200 import dist as jd

        self.torch, self.jd = torch, jd
        self.workload, self.rank, self.world, self.lib = workload, rank, world, lib
        self.dev = torch.device("cuda", local)
        self.desc, B, self.dtype_name = WORKLOADS[workload]
        self.B = batch or B
        self.model, self.img_size, self.text = build_model(workload, self.dtype_name)
        self.model.set_max_batch(self.B)
        self.dual = self.text is not None
        g = torch.Generator().manual_seed(1234 + rank)
        self.img_host = torch.randn(self.B, self.img_size, self.img_size, 3, generator=g, dtype=torch.float32).pin_memory()
        self.img_dev = self.img_host.to(self.dev)
        self.ids_host = self.ids_dev = None
        if self.dual:
            self.ids_host = synthetic_tokens(self.B, self.text[0], self.text[1], self.text[2], seed=4321 + rank).to(torch.int32).pin_memory()
            self.ids_dev = self.ids_host.to(self.dev)
            self.step_dev = lambda: self.model(self.img_dev, self.ids_dev)
            self.step_host = lambda: self.model(self.img_host, self.ids_host)
            # raw frames + token ids: what examples/clip_inference.py:35-38 hands its (host) processor; bytes over PCIe, front-end on the GPU
            from jimm_b200.preprocess import ImagePreprocessor

            self.u8_host = torch.randint(0, 256, (self.B, self.img_size, self.img_size, 3), generator=g, dtype=torch.uint8).pin_memory()
            self.model.set_preprocessor(ImagePreprocessor.clip(self.img_size) if workload == "clip_b32" else ImagePreprocessor.siglip(self.img_size))
            self.step_host_u8 = lambda: self.model(self.u8_host, self.ids_host)
        else:
            self.step_dev = lambda: self.model(self.img_dev)
            self.step_host = lambda: self.model(self.img_host)
            # raw frames: what examples/vit_inference.py:27-37 feeds its (host) image processor; here they cross PCIe as bytes and the
            # front-end (resize to the model size = identity window, rescale, normalise) runs on the GPU ahead of the tower
            from jimm_b200.preprocess import ImagePreprocessor

            self.u8_host = torch.randint(0, 256, (self.B, self.img_size, self.img_size, 3), generator=g, dtype=torch.uint8).pin_memory()
            self.model.set_preprocessor(ImagePreprocessor.vit(self.img_size))
            self.step_host_u8 = lambda: self.model(self.u8_host)

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed(self, fn, steps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dbg = [] if os.environ.get("JIMM_BENCH_DEBUG") else None
        for _ in range(steps):
            t0 = time.perf_counter()
            out = fn()
            if dbg is not None:
                dbg.append((time.perf_counter() - t0) * 1e3)
        e1.record()
        self.barrier()
        if dbg is not None:
            print(f"[bench debug] rank {self.rank} {getattr(fn, '__name__', 'fn')}: " + " ".join(f"{t:.2f}" for t in dbg), file=sys.stderr, flush=True)
        return self.jd.max_over_ranks(e0.elapsed_time(e1)), out

    @staticmethod
    def warm(fn, n=3):
        """Untimed calls with the SAME reference pattern as the timed loop (the previous result is still alive while the next call
        allocates its pinned result buffer): the first time two result buffers are needed the caching host allocator calls
        cudaHostAlloc, which synchronises the device -- a one-off 30 ms hiccup that belongs in the warm-up, not in step 2 of the timed
        region (seen with JIMM_BENCH_DEBUG=1)."""
        out = None
        for _ in range(n):
            out = fn()
        return out

    def rate(self, ms_total, steps):
        return self.world * self.B * steps / (ms_total * 1e-3)

    def e2e(self, steps, pipelined=True):
        """Host buffers through the public API: H2D + forward + D2H inside the timed region, synchronised every step."""
        out = {}
        self.warm(self.step_host)
        ms, out_h = self.timed(self.step_host, steps)
        f32 = {"value": self.rate(ms, steps), "ms_per_step": ms / steps,
               "h2d_bytes_per_step": self.img_host.numel() * 4 + (self.ids_host.numel() * 4 if self.dual else 0)}
        d2h = out_h.numel() * 4
        if self.step_host_u8 is None:
            out = {"value": f32["value"], "unit": "images/sec", "h2d_bytes_per_step": f32["h2d_bytes_per_step"], "d2h_bytes_per_step": d2h,
                   "ms_per_step": f32["ms_per_step"], "input": "pinned fp32 NHWC pixel values + int32 token ids", "sync": "every step"}
        else:
            self.warm(self.step_host_u8)
            ms8, _ = self.timed(self.step_host_u8, steps)
            out = {"value": self.rate(ms8, steps), "unit": "pairs/sec" if self.dual else "images/sec",
                   "h2d_bytes_per_step": self.u8_host.numel() + (self.ids_host.numel() * 4 if self.dual else 0), "d2h_bytes_per_step": d2h,
                   "ms_per_step": ms8 / steps, "sync": "every step",
                   "input": "pinned uint8 RGB frames" + (" + int32 token ids" if self.dual else "") + "; GPU image front-end (jimm_preproc_run) + tower(s) inside the timed region",
                   "fp32_input": f32}
            if pipelined and hasattr(self.model, "forward_async"):
                # the same loop with asynchronous dispatch, two calls in flight (every step still copies its inputs in and its result out)
                state = {"pending": None}

                def step_async():
                    nxt = self.model.forward_async(self.u8_host)
                    res = state["pending"].result() if state["pending"] is not None else None
                    state["pending"] = nxt
                    return res

                self.warm(step_async, 4)
                ms_pipe, _ = self.timed(step_async, steps)
                state["pending"].result()
                out["pipelined_depth2_value"] = self.rate(ms_pipe, steps)
        return out


def collective_leg(args, rank, world, local, lib):
    """N > 1: the dual-tower path with its one exchange step (embedding all-gather fused into the logits kernel over NVLink peer memory)."""
    import torch
    import torch.distributed as dist

    wl = os.environ.get("JIMM_BENCH_COLLECTIVE_WL") or ("siglip2_l16_512" if world >= 8 else "clip_b32")  # (override: dry-run the c5 leg on fewer GPUs)
    steps = args.steps
    bw = Bench(wl, 0, rank, world, local, lib)
    m, B = bw.model, bw.B
    m.set_comm("peer")
    for _ in range(3):
        bw.step_dev()
    torch.cuda.synchronize(bw.dev)
    ms, out = bw.timed(bw.step_dev, steps)
    host_step = bw.step_host_u8 or bw.step_host  # raw uint8 frames + token ids when the front-end is attached
    bw.warm(host_step)
    ms_h, _ = bw.timed(host_step, steps)
    n = m.native(B, require=True)
    # ---- the collective kernel alone: encoder outputs resident, CUDA events around `reps` back-to-back calls (every call carries its
    #      own cross-GPU flag barrier, so the ranks run it in lock-step), max over ranks
    ie, te = n.vision(bw.img_dev, encode=True), n.text(bw.ids_dev)
    reps = 50
    for _ in range(5):
        lg = n.comm_logits(ie, te)
    ms_k, lg = bw.timed(lambda: n.comm_logits(ie, te), reps)
    # per-call distribution (CUDA events around every call): the mean above includes whatever skew the two ranks' launch loops pick up
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    bw.barrier()
    evs[0].record()
    for i in range(reps):
        lg = n.comm_logits(ie, te)
        evs[i + 1].record()
    bw.barrier()
    per_call = sorted(evs[i].elapsed_time(evs[i + 1]) * 1e3 for i in range(reps))
    us_median = bw.jd.max_over_ranks(per_call[reps // 2])
    us_min, us_max = bw.jd.max_over_ranks(per_call[0]), bw.jd.max_over_ranks(per_call[-1])
    # NCCL baseline of the same exchange (normalise + all_gather_into_tensor + local logits), for context
    m.set_comm("nccl")
    for _ in range(5):
        m._distributed_logits(n, ie, te, B)
    ms_n, lg_nccl = bw.timed(lambda: m._distributed_logits(n, ie, te, B), reps)
    m.set_comm("peer")
    # ---- bit-identity with the single-GPU head (outside the timed region): gather the raw embeddings with NCCL, run the one-GPU head
    E = ie.shape[1]
    ie_all, te_all = torch.empty((world * B, E), device=bw.dev), torch.empty((world * B, E), device=bw.dev)
    dist.all_gather_into_tensor(ie_all, ie.contiguous())
    dist.all_gather_into_tensor(te_all, te.contiguous())
    # (the single-GPU head = l2_normalize + logits kernels of jimm_contrastive_logits, called through their per-kernel entry points because
    # the gathered text batch exceeds this handle's max_batch)
    def vp(t):
        return C.c_void_p(t.data_ptr())

    st = C.c_void_p(torch.cuda.current_stream(bw.dev).cuda_stream)
    ie_rows = ie_all[rank * B:(rank + 1) * B].contiguous()
    ni, nt = torch.empty_like(ie_rows), torch.empty_like(te_all)
    _lib_check = __import__("jimm_b200._lib", fromlist=["check"]).check
    _lib_check(lib.jimm_k_l2_normalize(vp(ie_rows), vp(ni), E, B, E, st))
    _lib_check(lib.jimm_k_l2_normalize(vp(te_all), vp(nt), E, world * B, E, st))
    scale = m.logit_scale.to(bw.dev).reshape(1).contiguous()
    bias = m.logit_bias.to(bw.dev).reshape(1).contiguous() if "logit_bias" in m._params else None
    single = torch.empty((B, world * B), dtype=torch.float32, device=bw.dev)
    _lib_check(lib.jimm_k_logits(vp(ni), vp(nt), vp(scale), vp(bias) if bias is not None else None, vp(single), B, world * B, E, world * B, st))
    same = torch.tensor([int(torch.equal(single, lg))], device=bw.dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    nccl_diff = bw.jd.max_over_ranks(float((lg_nccl - lg).abs().max()))
    bytes_per_peer = B * 2 * E * 4
    us = us_median
    egress = bytes_per_peer * (world - 1)
    return {
        "workload": WORKLOADS[wl][0] + f" x {world} GPUs = global batch {world * B}", "kernel": "comm_logits_kernel (csrc/comm.cu)",
        "reference_step": "the all-gather XLA inserts for image_features @ text_features.T under batch-sharded inputs "
                          "(models/clip.py:183-187, models/siglip.py:169-173, examples/clip_inference.py:41-44)",
        "value": bw.rate(ms, steps), "unit": "pairs/sec", "ms_per_step": ms / steps, "steps": steps,
        "e2e": {"value": bw.rate(ms_h, steps), "unit": "pairs/sec", "ms_per_step": ms_h / steps,
                "h2d_bytes_per_step": (bw.u8_host.numel() if bw.step_host_u8 else bw.img_host.numel() * 4) + bw.ids_host.numel() * 4,
                "d2h_bytes_per_step": B * world * B * 4, "input": "pinned uint8 RGB frames + int32 token ids" if bw.step_host_u8 else "pinned fp32 pixels + int32 token ids"},
        "us_per_call": us, "us_per_call_stat": "median of per-call CUDA-event times, max over ranks", "us_per_call_mean": ms_k / reps * 1e3,
        "us_per_call_min": us_min, "us_per_call_max": us_max, "calls_timed": reps, "bytes_sent_per_peer": bytes_per_peer, "peers": world - 1,
        "nvlink_egress_gbs": egress / (us * 1e-6) / 1e9, "nvlink_peak_gbs": 770.0, "nvlink_frac": egress / (us * 1e-6) / 1e9 / 770.0,
        "note": "latency-bound by construction: %.2f MiB per peer is %.1f us of NVLink time at 770 GB/s; the rest is normalise + flag barrier + "
                "the [B_local, B_global] logits tile" % (bytes_per_peer / 2**20, bytes_per_peer / 770e9 * 1e6),
        "nccl_allgather_us_per_call": ms_n / reps * 1e3, "max_abs_diff_vs_nccl_path": nccl_diff,
        "bit_identical_to_single_gpu": bool(same.item()), "collective_share_of_step": us * 1e-3 / (ms / steps),
    }


def run_ours(args):
    import torch

    from jimm_b200 import _lib, build
    from jimm_b200 import dist as jd

    rank, world, local = jd.init_from_env("nccl")
    if world != args.gpus and world > 1:
        args.gpus = world
    torch.cuda.set_device(local)
    build.build()
    lib = _lib.load()
    bw = Bench(args.workload, args.batch, rank, world, local, lib)
    B, dev = bw.B, bw.dev

    # ---- warm-up (also builds the native handle); the clock sampler is started first so that nvidia-smi is already streaming
    #      when the timed region begins (its start-up can take longer than a short timed region) ----
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        bw.step_dev()
    torch.cuda.synchronize(dev)
    native = bw.model.native(B)

    # ---- value: device-resident inputs ----
    l0 = lib.jimm_launch_count()
    sampler.mark_begin()
    ms_total, out = bw.timed(bw.step_dev, args.steps)
    sampler.mark_end()
    launches = lib.jimm_launch_count() - l0
    clocks = None
    if rank == 0:
        if sampler.proc is not None and sampler.in_window() == 0 and world == 1:
            # the region was shorter than the sampling period: keep the same load running (untimed) until a sample lands
            t_wait = time.time()
            while len([1 for t, _ in sampler.rows if t >= sampler.t1]) < 2 and time.time() - t_wait < 3.0:
                bw.step_dev()
                torch.cuda.synchronize(dev)
        clocks = sampler.stop()
    ms_step = ms_total / args.steps
    value = bw.rate(ms_total, args.steps)
    roofline = gemm_roofline(lib, native, bw.step_dev, args.steps, ms_step)
    e2e = bw.e2e(args.steps)
    peak_tf = roofline["peak"]

    # ---- N = 1 extras: the other headline workloads, K steps each ----
    extras = None
    if world == 1 and not args.no_extras and args.workload == "vit_b16":
        extras = {}
        steps = args.steps
        for wl in ("siglip_b16", "vit_l16_map"):
            bw = None  # free the previous model's workspace before the next one is built
            torch.cuda.empty_cache()
            try:
                bw = Bench(wl, 0, rank, world, local, lib)
                for _ in range(3):
                    bw.step_dev()
                torch.cuda.synchronize(dev)
                ms_x, _ = bw.timed(bw.step_dev, steps)
                v = bw.rate(ms_x, steps)
                rf = gemm_roofline(lib, bw.model.native(bw.B), bw.step_dev, steps, ms_x / steps)
                ex = bw.e2e(steps, pipelined=False)
                extras[wl] = {"workload": bw.desc, "value": v, "unit": "pairs/sec" if bw.dual else "images/sec", "ms_per_step": ms_x / steps, "steps": steps,
                              "dtype": {"float16": "f16", "bfloat16": "bf16"}[bw.dtype_name], "gflop_per_unit": GFLOP_PER_IMG[wl],
                              "model_tflops": v * GFLOP_PER_IMG[wl] / 1e3, "model_frac_of_peak": v * GFLOP_PER_IMG[wl] / 1e3 / peak_tf,
                              "e2e": ex, "gemm_tflops": rf["achieved"], "gemm_frac": rf["frac"], "gemm_share_of_step": rf["gemm_share_of_step"]}
            except Exception as e:  # the headline line must survive a failure of an extra leg (reported, not hidden)
                extras[wl] = {"error": f"{type(e).__name__}: {e}"[:400]}
        bw = None

    # ---- N > 1: the dual-tower leg with the fused NVLink exchange ----
    collective = None
    if world > 1 and not args.no_collective:
        bw = None
        torch.cuda.empty_cache()
        try:
            collective = collective_leg(args, rank, world, local, lib)
        except Exception as e:  # the headline line must survive a failure of the extra leg (reported, not hidden)
            collective = {"error": f"{type(e).__name__}: {e}"[:400]}

    # ---- CPU baseline (rank 0, N=1 only; bounded sample) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        # bounded sample of the same workload: ~12 s of host time, sized from a one-image probe
        probe_ips, _ = time_cpu(args.workload, 1, 1, 1)
        cb = max(1, min(16, int(probe_ips * 2.0)))
        csteps = args.cpu_steps if args.cpu_steps > 0 else max(2, min(60, int(12.0 * probe_ips / cb)))
        ips, _ = time_cpu(args.workload, cb, csteps, 1)
        cpu = {"value": ips, "unit": "images/sec", "cores": cpu_threads(), "host_cores": os.cpu_count() or 1, "kind": "port",
               "sample": f"{cb} images/step x {csteps} steps, oracle/jimm_oracle.py torch-CPU fp32 (jimm semantics)"}

    if args.dump_outputs:
        # what a caller of the headline loop receives from its last timed step: logits, or the pooled features of a bare tower
        name = "features" if args.workload == "vit_l16_map" else "logits"
        for path in dump_outputs(args.dump_outputs, {name: out}, rank, world):
            print(f"bench: wrote {path}", file=sys.stderr, flush=True)

    if rank == 0:
        gflop = GFLOP_PER_IMG[args.workload]
        desc, _, dtype_name = WORKLOADS[args.workload]
        line = {
            "metric": "images/sec", "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"float16": "f16", "bfloat16": "bf16", "float32": "tf32"}[dtype_name], "data": "synthetic",
            "config": {"workload": desc, "per_gpu_batch": B, "global_batch": world * B, "parallelism": f"dp{world}",
                       "l2_policy": "inputs_larger_than_L2 (154 MB fp32 images; >1 GB of activations streamed per step)",
                       "gflop_per_image": gflop},
            "model_tflops": value * gflop / 1e3, "model_frac_of_peak": value * gflop / 1e3 / (peak_tf * world),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        }
        if extras is not None:
            line["extra_workloads"] = extras
        if collective is not None:
            line["collective"] = collective
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="vit_b16", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch override")
    ap.add_argument("--cpu-batch", type=int, default=4)
    ap.add_argument("--cpu-steps", type=int, default=0, help="0 = size the CPU sample for ~12 s")
    ap.add_argument("--cpu-batch-fixed", action="store_true", help="reference arm: use --cpu-batch instead of sizing it from a probe")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N=1: skip the SigLIP-B/16@256 and ViT-L/16@384 legs")
    ap.add_argument("--no-collective", action="store_true", help="N>1: skip the dual-tower leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
