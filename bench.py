"""bench.py -- images/sec of the PerspectiveFields inference hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config C2|C3|C4|C5|P360]     # this repo's CUDA path
    python bench.py --impl reference [...]                                              # the reference algorithm on the host CPU cores
    python bench.py --dump-outputs DIR [...]                                            # + the last timed step's results as DIR/<key>.npy

A step is one pass of the hot path over one batch of synthetic input.  Configurations (BASELINE.json `configs`, SURVEY.md 8d):
  C2 (default, the configuration the metric is quoted on): ``Paramnet-360Cities-edina-centered``, 32 x 640x480 per GPU
  C3: ``Paramnet-360Cities-edina-uncentered`` (principal-point head), 64 x 512x512
  C4: ``PersNet_Paramnet-GSV-uncentered``, 32 x 640x480 per GPU (256 over 8 GPUs) -- the multi-GPU configuration
  C5: resolution sweep 320x240 / 640x480 / 1024x768 / 2048x1536, batch 8: HBM roofline of the pre/post-processing per resolution
  P360: ``PersNet-360Cities`` (73 / 180-class heads), 32 x 640x480, default (logits returned) and "decode_only" mode (SURVEY 8f-3)
Inputs are uniform-random uint8 BGR images; weights a seeded synthetic checkpoint (trained weights are not available offline).

Multi-GPU: one process per GPU (torchrun).  Each rank runs its own shard of the global batch -- independent images, no
data-path collective ("weak" scaling); `value` is that number.  In addition (N > 1) the `gather` object reports the same K steps
through ``dist.inference_batch_sharded``: every rank passes the whole list, results are gathered to rank 0's device with grouped
ncclSend/ncclRecv (``pf_gather``) on a side stream INSIDE the timed region -- what one ``inference_batch(list of N*32)`` call on a
multi-GPU box does.

Prints ONE JSON line on rank 0:  value = whole-job images/s with inputs resident in HBM (CUDA events, max over ranks),
e2e = the same through the public API from host numpy arrays incl. H2D of the inputs and D2H of every returned tensor,
roofline = achieved algorithmic FLOP/s of the dominant kernel measured with CUDA events vs the measured bf16 peak,
roofline_post = achieved GB/s of the HBM-bound write-out stage, cpu_baseline = the oracle port of the reference timed on the host.
"""
import argparse
import ctypes
import gc
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "images/sec at 640x480 (Paramnet-360Cities-edina), 1/2/4/8xB200 vs ref CPU"
CONFIGS = {
    "C2": dict(version="Paramnet-360Cities-edina-centered", batch=32, sizes=[(480, 640)],
               workload="C2: Paramnet-360Cities-edina-centered, batch=32 640x480 synthetic uint8 BGR per GPU, seeded synthetic checkpoint"),
    "C3": dict(version="Paramnet-360Cities-edina-uncentered", batch=64, sizes=[(512, 512)],
               workload="C3: Paramnet-360Cities-edina-uncentered (principal-point head), batch=64 512x512 synthetic uint8 BGR per GPU, seeded synthetic checkpoint"),
    "C4": dict(version="PersNet_Paramnet-GSV-uncentered", batch=32, sizes=[(480, 640)],
               workload="C4: PersNet_Paramnet-GSV-uncentered, 32 x 640x480 synthetic uint8 BGR per GPU (256 over 8 GPUs), seeded synthetic checkpoint"),
    "C5": dict(version="Paramnet-360Cities-edina-centered", batch=8, sizes=[(240, 320), (480, 640), (768, 1024), (1536, 2048)],
               workload="C5: resolution sweep 320x240 / 640x480 / 1024x768 / 2048x1536, batch=8, Paramnet-360Cities-edina-centered, seeded synthetic checkpoint"),
    "P360": dict(version="PersNet-360Cities", batch=32, sizes=[(480, 640)],
                 workload="P360: PersNet-360Cities (73 / 180-class heads), batch=32 640x480 synthetic uint8 BGR per GPU, seeded synthetic checkpoint"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the configuration's)")
    ap.add_argument("--cpu-sample", type=int, default=8, help="images in the bounded CPU-baseline sample")
    ap.add_argument("--micro-batch", type=int, default=32, help="images per micro-batch of the gather-inclusive multi-GPU leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile-passes", action="store_true", help="skip the roofline / per-kernel passes (A/B timing runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step (rank 0's shard) as DIR/<key>.npy")
    return ap.parse_args()


class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region (B200_PROFILING.md recipe), read through NVML from the
    main thread once all K steps have been enqueued, repeatedly until the end event completes (the GPU is busy with the queued
    steps; sampling between the enqueues starved the GPU on boxes where one NVML call takes ~40 ms).
    A concurrent poller -- an `nvidia-smi -lms` child or an NVML thread -- measurably slowed the launches it was observing."""

    def __init__(self, index):
        self.index, self.rows, self.nvml = index, [], None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    def sample(self):
        try:
            if self.nvml is not None:
                n = self.nvml
                sm = n.nvmlDeviceGetClockInfo(self.h, n.NVML_CLOCK_SM)
                try:
                    r = n.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                reasons = [name for name, bit in (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20),
                                                  ("hw_thermal_slowdown", 0x40)) if r & bit]
                self.rows.append((sm, self.max_sm, reasons))
            else:
                q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                     "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
                c = [x.strip() for x in subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                                       capture_output=True, text=True).stdout.strip().split(",")]
                reasons = [nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[2:6]) if v.lower().startswith("active")]
                self.rows.append((float(c[0]), float(c[1]), reasons))
        except Exception:
            pass

    def stop(self):
        sm = sorted(r[0] for r in self.rows)
        reasons = sorted({x for r in self.rows for x in r[2]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.rows[0][1] if self.rows else None, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


def physical_cores():
    """Threads for the CPU reference: one per physical core (torch's own default when OMP_NUM_THREADS is unset).  Using every
    hyper-thread (128 on this pool's hosts) makes ATen's CPU kernels ~10x SLOWER, which would only flatter the GPU number."""
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
        if n:
            return int(n)
    except Exception:
        pass
    return max(1, (os.cpu_count() or 2) // 2)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def make_images(cfg, batch, seed):
    from oracle import weights_gen as wg   # synthetic inputs / checkpoint generator (test infrastructure)

    h, w = cfg["sizes"][0]
    return wg.synth_images(batch, h, w, seed)


def cpu_reference_images_per_s(cfg, n_images, repeats):
    """The reference algorithm (oracle port, oracle/model.py == reference ATen calls) on the host cores: one full-sample warm-up,
    then `repeats` timed passes of the SAME sample; median."""
    import torch

    from oracle import model as om
    from oracle import weights_gen as wg

    torch.set_num_threads(physical_cores())
    sd = wg.synth_state_dict(cfg["version"], 0)
    imgs = make_images(cfg, n_images, 0)
    om.inference_batch(sd, cfg["version"], imgs)  # warm-up on the whole sample (thread pool, allocator, oneDNN primitives)
    ts = []
    for _ in range(repeats):
        t = time.perf_counter()
        om.inference_batch(sd, cfg["version"], imgs)
        ts.append(time.perf_counter() - t)
    ts.sort()
    return n_images / ts[len(ts) // 2], torch.get_num_threads(), [round(n_images / t, 3) for t in ts]


def workload_config(args, cfg, B, world):
    return {"workload": cfg["workload"], "global_batch": B * world,
            "parallelism": f"dp{world} (independent images, no data-path collective)",
            "l2": "256 MiB flush write between timed steps; per-step working set (activations of the batch) >> 126 MB L2"}


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: the reference is pure Python
    and /root/reference does not exist on the GPU box) on all physical host cores; each step = inference_batch of a bounded
    sample of the workload (`cpu_baseline.sample`); `config` is this repo's arm's."""
    if rank != 0:
        return
    import torch

    from oracle import model as om
    from oracle import weights_gen as wg

    cfg = CONFIGS[args.config]
    B = args.batch or cfg["batch"]
    torch.set_num_threads(physical_cores())     # torchrun exports OMP_NUM_THREADS=1: set the pool size explicitly
    sd = wg.synth_state_dict(cfg["version"], 0)
    n = min(args.cpu_sample, B)
    imgs = make_images(cfg, n, 0)
    for _ in range(min(args.warmup, 1)):
        om.inference_batch(sd, cfg["version"], imgs)
    per_step = []
    for _ in range(args.steps):
        t = time.perf_counter()
        res = om.inference_batch(sd, cfg["version"], imgs)
        per_step.append(time.perf_counter() - t)
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    dt = sum(per_step)
    v = n * args.steps / dt
    sample = (f"{n} of the {B} images of the step's batch per step ({args.steps} steps, 1 warm-up on the same sample), torch CPU fp32, "
              f"{torch.get_num_threads()} threads = physical cores of '{cpu_model()}' ({os.cpu_count()} logical); per-step img/s min/median/max = "
              f"{n / max(per_step):.2f}/{n / sorted(per_step)[len(per_step) // 2]:.2f}/{n / min(per_step):.2f}")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1000, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, cfg, B, args.gpus),
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample, "cpu": cpu_model()},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


class Bench:
    """Shared state of the timed legs of one model / workload."""

    def __init__(self, args, cfg, dev, rank, world, model_kwargs=None):
        import torch
        import torch.distributed as dist

        import pf_test_util as U
        from perspectivefields_b200 import _native

        self.torch, self.dist, self.N = torch, dist, _native
        self.args, self.cfg, self.dev, self.rank, self.world = args, cfg, dev, rank, world
        self.model, _sd = U.make_model(cfg["version"], seed=0, device=dev, model_kwargs=model_kwargs)
        self.eng = self.model._get_engine()
        for kv in filter(None, os.environ.get("PF_BENCH_OPTS", "").split(",")):   # A/B runs of engine options, e.g. PF_BENCH_OPTS=phase_conv1=0
            k, v = kv.split("=")
            self.model.set_option(k, int(v))
        self.L = _native.lib()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > L2 (126 MB)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, ms):
        t = self.torch.tensor([ms], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def resident_leg(self, imgs, steps, warmup, sampler=None, trace=False, dump_dir=None):
        """K steps with the inputs already in HBM: flush L2, pf_forward on the staged blob.  Returns (ms of the timed region on this
        rank, kernel launches, host enqueue ms per step).  ``dump_dir``: write the last step's results there (dump_outputs)."""
        torch = self.torch
        B = len(imgs)
        heights, widths = [im.shape[0] for im in imgs], [im.shape[1] for im in imgs]
        blob, offsets = self.eng.stage_images(imgs)
        torch.cuda.synchronize(self.dev)
        out = None
        for _ in range(warmup):    # same sequence as a timed step (flush, forward, result rebinding)
            self.flush.fill_(1)
            out = self.eng.forward(B, heights, widths, blob=blob, offsets=offsets)
        gc.collect()
        self.barrier()
        l0 = self.L.pf_kernel_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        for _ in range(steps):
            self.flush.fill_(1)  # L2 flush between timed iterations (inside the timed region: ~0.1 ms of ~20)
            out = self.eng.forward(B, heights, widths, blob=blob, offsets=offsets)
        e1.record()
        host_ms = (time.perf_counter() - t0) * 1000 / steps
        if sampler is not None:
            # clock samples DURING the timed region: the host is ahead of the GPU here (all K steps are queued), so the NVML calls
            # (tens of ms each on some boxes) overlap the GPU work instead of delaying launches
            sampler.sample()
            while not e1.query() and len(sampler.rows) < 64:
                sampler.sample()
        self.barrier()
        if dump_dir is not None:
            dump_outputs(self.model.assemble_raw(out), dump_dir)
        del out
        return e0.elapsed_time(e1), self.L.pf_kernel_launch_count() - l0, host_ms, (blob, offsets, heights, widths)

    def profile_passes(self, staged, steps):
        """Roofline pass (CUDA-event pair around every GEMM-engine launch) and per-kernel pass (around EVERY launch): the same K
        steps again, kept out of the `value` region because the event records perturb it."""
        torch, L, N = self.torch, self.L, self.N
        blob, offsets, heights, widths = staged
        B = len(heights)
        N.check(L.pf_profile_enable(self.eng.handle, 300 * steps))
        self.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(steps):
            self.flush.fill_(1)
            self.eng.forward(B, heights, widths, blob=blob, offsets=offsets)
        g1.record()
        self.barrier()
        prof_ms = g0.elapsed_time(g1)
        prof = (ctypes.c_double * 21)()
        N.check(L.pf_profile_read(self.eng.handle, prof))
        N.check(L.pf_profile_enable(self.eng.handle, 0))
        N.check(L.pf_profile_kernels_enable(self.eng.handle, 700 * steps))
        self.barrier()
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(steps):
            self.flush.fill_(1)
            self.eng.forward(B, heights, widths, blob=blob, offsets=offsets)
        k1.record()
        self.barrier()
        buf = ctypes.create_string_buffer(1 << 16)
        nbytes = N.check(L.pf_profile_kernels_read(self.eng.handle, buf, len(buf)))
        N.check(L.pf_profile_kernels_enable(self.eng.handle, 0))
        per_kernel = {}
        for line in buf.raw[:nbytes].decode().splitlines()[1:]:
            name, cnt, kms = line.rsplit(",", 2)
            per_kernel[name] = {"ms_per_step": round(float(kms) / steps, 4), "launches_per_step": int(cnt) / steps}
        per_kernel["_pass_ms_per_step"] = round(k0.elapsed_time(k1) / steps, 3)
        return list(prof), prof_ms, per_kernel

    def e2e_leg(self, imgs, steps, warmup):
        """End to end through the public API: host arrays in (pinned staging + H2D inside), every returned tensor read back to pinned
        host memory on a side stream (overlapping the next step's forward), all inside the timed region."""
        torch = self.torch
        B = len(imgs)
        res = self.model.inference_batch(imgs)
        keys = [k for k, v in res[0].items() if not isinstance(v, str)]
        host = [{k: torch.empty((B,) + tuple(res[0][k].shape), dtype=torch.float32).pin_memory() for k in keys} for _ in range(2)]
        d2h_bytes = sum(v.numel() * 4 for v in host[0].values())
        h2d_bytes = sum(im.size for im in imgs)
        del res
        copy_stream = torch.cuda.Stream(device=self.dev)
        pending = []
        it = [0]

        def step():
            r = self.model.inference_batch(imgs)
            done = torch.cuda.Event()
            done.record()
            bufs = host[it[0] % 2]
            it[0] += 1
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done)
                for i, d in enumerate(r):
                    for k in keys:
                        bufs[k][i].copy_(d[k], non_blocking=True)
            if len(pending) >= 2:
                old_ev, old_r = pending.pop(0)
                old_ev.synchronize()            # the buffers about to be reused have been filled ...
                del old_r                       # ... and only now are that step's device results released
            ev = torch.cuda.Event()
            ev.record(copy_stream)
            pending.append((ev, r))

        for _ in range(max(warmup, 1)):
            step()
        self.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        tw = time.perf_counter()
        f0.record()
        for _ in range(steps):
            step()
        torch.cuda.current_stream(self.dev).wait_stream(copy_stream)   # the last read-back is inside the timed region
        f1.record()
        self.barrier()
        wall_ms = (time.perf_counter() - tw) * 1000
        pending.clear()
        return max(f0.elapsed_time(f1), wall_ms), h2d_bytes, d2h_bytes


DUMP_MAX_ELEMENTS = 1 << 21   # per key (8 MiB of float32): the four field keys of a step stay below 64 MB in all


def dump_outputs(results, dirname):
    """The result dictionaries of ``inference_batch`` (what a caller of the timed path receives) as DIR/<key>.npy, float32,
    one file per tensor key with the images stacked on a leading axis (the scalar camera parameters become [n] vectors).  A key
    of more than DUMP_MAX_ELEMENTS elements is written flattened and sampled: the elements at sorted flat indices drawn with a
    fixed seed from its size alone, so that the files of two builds run with the same arguments compare element for element."""
    import numpy as np
    import torch

    os.makedirs(dirname, exist_ok=True)
    for key, v in results[0].items():
        if isinstance(v, str):
            continue
        t = torch.stack([r[key] for r in results])
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), DUMP_MAX_ELEMENTS))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(dirname, key + ".npy"), t.float().cpu().numpy())


def roofline_objects(args, B, prof, prof_ms, ms, per_kernel, heights, widths, peaks, write_peak=None):
    peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    traffic, traffic_src = None, None
    for name in ("r02_ncu_dominant_kernel.json", "r01_ncu_dominant_kernel.json"):
        try:   # DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (profiles/)
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            traffic, traffic_src = t["dram_bytes_per_launch"], t["source"]
            break
        except Exception:
            pass
    names = {5: "gemm_tma_kernel<BN,GEMM> (persistent TMA -> tcgen05.mma kind::f16 -> TMEM, bf16x3 split precision, 128 x BN tiles: every Linear / 1x1 / patchified conv)",
             6: "gemm_tma_kernel<BN,HALO> (persistent TMA halo -> tcgen05.mma kind::f16 -> TMEM, bf16x3 split precision, 3x3 conv, 16x8-pixel x BN tiles)"}
    cfgs = [c for c in range(7) if prof[3 * c + 2] > 0]
    gemm_ms = sum(prof[3 * c] for c in cfgs)
    gemm_flops = sum(prof[3 * c + 1] for c in cfgs)
    dom = max(cfgs, key=lambda c: prof[3 * c])
    dom_ms, dom_flops, dom_n = prof[3 * dom], prof[3 * dom + 1], prof[3 * dom + 2]
    achieved = dom_flops / (dom_ms / 1000.0) / 1e12 if dom_ms > 0 else None
    roofline = {
        "bound": "tensor", "kernel": names.get(dom, str(dom)),
        "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": (achieved / peak_tf) if achieved else None,
        "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
        "note": "achieved = algorithmic 2*M*N*K FLOPs / CUDA-event time of this kernel's launches, measured live in a second pass of the same K steps "
                "(event pairs on the launch stream around every GEMM launch; kept out of the `value` region); every product costs "
                "3 bf16 MMAs (lo*hi + hi*lo + hi*hi) to meet the 1e-3 fp32 tolerance, so the ceiling of this scheme is peak/3 (frac 0.33)",
        "launches_per_step": dom_n / args.steps, "ms_per_step": dom_ms / args.steps,
        "all_gemm_ms_per_step": gemm_ms / args.steps, "all_gemm_share_of_step": gemm_ms / ms if ms > 0 else None,
        "profiled_pass_ms_per_step": prof_ms / args.steps,
        "all_gemm_tflops": gemm_flops / (gemm_ms / 1000.0) / 1e12 if gemm_ms > 0 else None,
        "gflop_per_image_gemm": gemm_flops / (args.steps * B) / 1e9,
        "per_engine": {names[c].split(" (")[0]: {"ms_per_step": prof[3 * c] / args.steps, "tflops": prof[3 * c + 1] / (prof[3 * c] / 1000.0) / 1e12,
                                                 "launches_per_step": prof[3 * c + 2] / args.steps} for c in cfgs},
    }
    return roofline, post_roofline(per_kernel, heights, widths, peaks, write_peak)


def post_roofline(per_kernel, heights, widths, peaks, write_peak=None):
    """HBM-bound tail of the path (SURVEY 8d: the "decode-head" HBM roofline applies to the write-out stage): resample of the
    three 320x320 fields to the original sizes + normalise / asin.  Algorithmic bytes = 4*(3*320*320 read + 3*H*W written) per image."""
    pk = per_kernel.get("postprocess_kernel")
    if not pk or pk["ms_per_step"] <= 0:
        return None
    post_bytes = sum(4 * (3 * 320 * 320 + 3 * int(h_) * int(w_)) for h_, w_ in zip(heights, widths))
    hbm_peak = peaks.get("hbm_gbs") or 6500.0
    gbps = post_bytes / (pk["ms_per_step"] / 1000.0) / 1e9
    r = {"bound": "hbm", "kernel": "postprocess_kernel (bilinear resample to (H,W) + F.normalize / asin, all images of the batch in one launch)",
         "achieved": gbps, "peak": hbm_peak, "unit": "GB/s", "frac": gbps / hbm_peak, "bytes_per_step": post_bytes,
         "ms_per_step": pk["ms_per_step"], "size": f"{widths[0]}x{heights[0]} x {len(heights)}",
         "note": "in-pipeline CUDA-event time of the per-kernel pass (includes ~2-4 us of event overhead per launch); `peak` is the measured "
                 "COPY bandwidth (read + write bytes); the kernel's traffic is 75 % writes, and `write_peak` is this GPU's measured write-only "
                 "bandwidth (torch fill_ of 1 GiB), the bound that applies to them"}
    if write_peak:
        wbytes = sum(12 * int(h_) * int(w_) for h_, w_ in zip(heights, widths))
        r["write_peak"] = write_peak
        r["write_gbs"] = wbytes / (pk["ms_per_step"] / 1000.0) / 1e9
        r["frac_of_write_peak"] = r["write_gbs"] / write_peak
    return r


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def measured_write_peak(dev):
    """Pure-WRITE bandwidth of this GPU's HBM (GB/s), measured live the way MEASURED_PEAKS.json measures the copy peak: the better
    of torch ``fill_`` and a 16-byte streaming-store kernel (pf_op_fill_stream) over 1 GiB, best of 4 each, CUDA events.  The copy peak counts read + write bytes; a kernel that only writes (the
    post-process / camera-field write-out) cannot exceed this number, which on this pool's B200s is well below half the copy peak."""
    import torch

    from perspectivefields_b200 import _native

    L = _native.lib()
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    best = 0.0
    for fn in (lambda: a.fill_(3), lambda: _native.check(L.pf_op_fill_stream(a.data_ptr(), a.numel() // 4, 1.0, st))):   # torch's fill and 16-byte streaming stores
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize(dev)
            best = max(best, a.numel() / e0.elapsed_time(e1) / 1e6)
    del a
    return best


def camera_fields_roofline(dev, heights, widths, peaks, steps, write_peak=None):
    """Row f-1 (camera parameters -> dense fields): 12 B of stores per pixel.  The launch sequence of one call is captured in a
    CUDA graph and replayed, so that the CUDA-event time is the kernels' (the Python + descriptor build of a call costs more than
    the kernel at small sizes); falls back to timing back-to-back calls."""
    import torch

    from perspectivefields_b200 import panocam

    n = len(heights)
    args_ = ([0.8] * n, heights, widths, [0.3] * n, [0.1] * n, [0.02] * n, [-0.03] * n)
    panocam.camera_fields(*args_, device=dev)
    torch.cuda.synchronize(dev)
    reps = max(steps, 10)
    how = "CUDA graph replay of one call's launches"
    try:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            panocam.camera_fields(*args_, device=dev)
        torch.cuda.current_stream(dev).wait_stream(side)
        with torch.cuda.graph(g):
            out = panocam.camera_fields(*args_, device=dev)
        run = g.replay
    except Exception as ex:   # capture not possible: time whole calls
        how = f"back-to-back calls incl. host work ({type(ex).__name__})"
        run = lambda: panocam.camera_fields(*args_, device=dev)
    run()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    nbytes = 12 * sum(int(h) * int(w) for h, w in zip(heights, widths))
    hbm_peak = peaks.get("hbm_gbs") or 6500.0
    r = {"kernel": "camera_fields_kernel", "ms": ms, "bytes": nbytes, "achieved": nbytes / ms / 1e6, "peak": hbm_peak, "unit": "GB/s",
         "frac": nbytes / ms / 1e6 / hbm_peak, "timing": how}
    if write_peak:
        r["write_peak"] = write_peak
        r["frac_of_write_peak"] = nbytes / ms / 1e6 / write_peak
    return r


def gather_leg(b, imgs_rank, steps, warmup, micro_batch):
    """N > 1: K steps of ``dist.inference_batch_sharded`` -- every rank holds the WHOLE list (its own shard's images are real, the
    others' are same-shape placeholders it never touches), results gathered to rank 0's device with pf_gather (grouped ncclSend /
    ncclRecv on a side stream) inside the timed region."""
    import numpy as np

    torch = b.torch
    from perspectivefields_b200 import dist as pfdist

    world, rank = b.world, b.rank
    B = len(imgs_rank)
    placeholder = np.zeros_like(imgs_rank[0])
    full = [placeholder] * (world * B)
    full[rank * B:(rank + 1) * B] = imgs_rank
    tr = pfdist.PfCommTransport(b.dev)
    res, ev, prev = None, None, None
    for _ in range(max(warmup, 1)):
        res = pfdist.inference_batch_sharded(b.model, full, gather_to=0, micro_batch=micro_batch, transport=tr)
    b.barrier()
    moved0 = tr.bytes_moved
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tw = time.perf_counter()
    e0.record()
    for _ in range(steps):
        b.flush.fill_(1)
        # pipelined calls (wait=False): the gather of step k overlaps the forward of step k+1; the results of step k are released
        # only after their event has completed (two steps in flight), and the last gather is inside the timed region
        res, ev = pfdist.inference_batch_sharded(b.model, full, gather_to=0, micro_batch=micro_batch, transport=tr, wait=False)
        if prev is not None:
            prev[1].synchronize()
        prev = (res, ev)
    torch.cuda.current_stream(b.dev).wait_event(ev)
    e1.record()
    b.barrier()
    res = prev[0]
    prev = None
    wall_ms = (time.perf_counter() - tw) * 1000
    ms = b.max_over_ranks(max(e0.elapsed_time(e1), wall_ms))
    moved = tr.bytes_moved - moved0
    n_back = len(res) if rank == 0 else None
    del res
    tr.close()
    out = {"value": world * B * steps / (ms / 1000.0), "unit": "images/s", "ms_per_step": ms / steps, "micro_batch": micro_batch,
           "images_per_call": world * B, "transport": "pf_gather: grouped ncclSend/ncclRecv from libpf_b200.so on a side stream, inside the timed region; calls pipelined (the "
                        "gather of step k overlaps the forward of step k+1, receives posted after the root's own forward)"}
    if rank == 0:
        out.update({"bytes_received_per_step_rank0": moved / steps, "achieved_gbs_into_rank0": moved / (ms / 1000.0) / 1e9,
                    "results_on_rank0": n_back,
                    "note": "achieved_gbs is bytes / whole step time (the transfers overlap the forward; NVLink 5 peak is 900 GB/s per direction)"})
    return out


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    cfg = CONFIGS[args.config]
    B = args.batch or cfg["batch"]
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    peaks = load_peaks()
    extra = {}
    write_peak = measured_write_peak(dev)
    extra["hbm_write_gbs_measured"] = write_peak

    b = Bench(args, cfg, dev, rank, world)
    imgs = make_images(cfg, B, 1000 + rank)   # each rank owns its shard of the global batch
    sampler = ClockSampler(local)   # NVML is initialised before the warm-up: its start-up must not leave the GPU idle in front of the timed steps
    # the cyclic garbage collector is off inside the timed regions (as timeit does): a generation-2 pass over the interpreter's
    # ~10^6 objects is a 10-100 ms host stall, longer than the two steps of work the launch queue holds
    gc.collect()
    gc.disable()

    # ---------------- leg 1: inputs resident in HBM ("value") ------------------------------------------------
    ms, launches, host_ms, staged = b.resident_leg(imgs, args.steps, args.warmup, sampler,
                                                   dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop()
    ms_max = b.max_over_ranks(ms)
    value = world * B * args.steps / (ms_max / 1000.0)
    roofline = roofline_post = None
    per_kernel = {}
    if not args.no_profile_passes:
        prof, prof_ms, per_kernel = b.profile_passes(staged, args.steps)
        roofline, roofline_post = roofline_objects(args, B, prof, prof_ms, ms, per_kernel, staged[2], staged[3], peaks, write_peak)
    del staged

    # ---------------- leg 2: end to end through the public API, host arrays in, results read back to the host -----
    e2e_ms, h2d_bytes, d2h_bytes = b.e2e_leg(imgs, args.steps, args.warmup)
    e2e_value = world * B * args.steps / (b.max_over_ranks(e2e_ms) / 1000.0)

    # ---------------- N > 1: the same steps with the results gathered to rank 0 over NVLink (inside the timed region) ----------
    if world > 1:
        extra["gather"] = gather_leg(b, imgs, args.steps, args.warmup, args.micro_batch)

    # ---------------- C5: resolution sweep (pre/post-processing bytes are the only thing that changes) ---------------------
    if args.config == "C5" and rank == 0:
        from oracle import weights_gen as wg
        sweep = []
        for (h, w) in cfg["sizes"]:
            im = wg.synth_images(B, h, w, 7)
            ms_r, _, _, st = b.resident_leg(im, args.steps, args.warmup)
            row = {"size": f"{w}x{h}", "batch": B, "images_per_s": B * args.steps / (ms_r / 1000.0), "ms_per_step": ms_r / args.steps}
            if not args.no_profile_passes:
                _, _, pk = b.profile_passes(st, args.steps)
                row["roofline_post"] = post_roofline(pk, st[2], st[3], peaks, write_peak)
                pre = pk.get("preprocess_kernel")
                if pre:
                    pre_bytes = B * (3 * h * w + 16 * 320 * 320)
                    row["preprocess"] = {"ms_per_step": pre["ms_per_step"], "bytes_per_step": pre_bytes, "achieved_gbs": pre_bytes / pre["ms_per_step"] / 1e6}
            row["camera_fields"] = camera_fields_roofline(dev, [h] * B, [w] * B, peaks, max(args.steps, 5), write_peak)
            del st
            sweep.append(row)
        extra["resolution_sweep"] = sweep
    elif rank == 0 and world == 1:
        h, w = cfg["sizes"][0]
        extra["roofline_camera_fields"] = camera_fields_roofline(dev, [h] * B, [w] * B, peaks, max(args.steps, 5), write_peak)

    # ---------------- P360: the classification variant without logits (option "decode_only") -------------------------------
    if args.config == "P360":
        b2 = Bench(args, cfg, dev, rank, world, model_kwargs={"logits": False})
        ms2, launches2, _, st2 = b2.resident_leg(imgs, args.steps, args.warmup)
        v2 = world * B * args.steps / (b2.max_over_ranks(ms2) / 1000.0)
        del st2
        e2, h2d2, d2h2 = b2.e2e_leg(imgs, args.steps, args.warmup)
        extra["decode_only"] = {"value": v2, "unit": "images/s", "ms_per_step": b2.max_over_ranks(ms2) / args.steps,
                                "e2e": {"value": world * B * args.steps / (b2.max_over_ranks(e2) / 1000.0), "unit": "images/s", "h2d_bytes_per_step": h2d2,
                                        "d2h_bytes_per_step": d2h2},
                                "gpu_launches": int(launches2),
                                "note": "PerspectiveFields(version, logits=False): pred_gravity / pred_latitude are the decoded fields; the 73 / 180 logit "
                                        "tensors (103.6 MB per image) are never written"}
    gc.enable()

    # ---------------- CPU baseline: oracle port of the reference on the host cores (rank 0, N = 1 only) ---------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n = min(args.cpu_sample, B)
        v, threads, reps = cpu_reference_images_per_s(cfg, n, 3)
        cpu = {"value": v, "unit": "images/s", "cores": threads, "kind": "port", "cpu": cpu_model(), "repeats_images_per_s": reps,
               "sample": f"inference_batch of {n} of the workload's images, one warm-up pass on the same sample, median of 3, torch CPU fp32, one thread per physical core (host has {os.cpu_count()} logical cores)"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 via 3x bf16 split MMA, fp32 accumulate", "data": "synthetic",
            "config": workload_config(args, cfg, B, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes},
            "gpu_launches": int(launches),
            "host_enqueue_ms_per_step": host_ms,
            "roofline": roofline,
            "roofline_post": roofline_post,
            "per_kernel": per_kernel,
            "cpu_baseline": cpu,
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
