#!/usr/bin/env python
"""bench.py -- SmaAt-UNet forward frames/sec on B200 (BASELINE.json metric), one JSON line.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--mode tf32x3|tf32|fp32] [--dump-outputs DIR]

* own arm (``--impl b200``): N ranks (torchrun for N>1), each with the full model and its own
  shard of B=32 synthetic 12x288x288 frames per step (weak scaling, eval forward has no
  collective -- SURVEY 8e).  ``value`` = frames/s with inputs resident in HBM (CUDA-graph replay,
  CUDA events, barrier + synchronize both sides, max over ranks); ``e2e`` = the same through
  ``InferenceSession.submit/collect`` with pinned HOST buffers (H2D + D2H inside the timed region);
  ``roofline`` = the depthwise kernel (the metric's named kernel) timed live with CUDA events,
  algorithmic bytes / time vs MEASURED_PEAKS.json; ``cpu_baseline`` = the oracle's torch CPU port
  on a bounded sample (rank 0, N=1 only).
* reference arm (``--impl reference``): the reference's CPU path (oracle/torch_port.py: same
  ATen/oneDNN kernels as the reference modules; /root/reference is not on the GPU box) on all
  host threads, each step a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
B_PER_GPU, C_IN, SIZE = 32, 12, 288


def note(msg):
    """Progress marker on stderr (stdout carries only the JSON line)."""
    if int(os.environ.get("RANK", "0")) == 0:
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def peaks():
    """(HBM GB/s, dense tf32 TFLOP/s, source).  tf32 tensor peak = half the measured cuBLAS bf16 burst figure (a kernel
    timed launch by launch); nominal ratio bf16:tf32 = 2:1 (B200_PROFILING.md)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]) / 2.0, "measured (MEASURED_PEAKS.json; tf32 = bf16 burst / 2)"
    return 6650.0, 1590.0 / 2.0, "fallback (B200_PROFILING.md; tf32 = bf16 / 2)"


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def ncu_traffic(kernel_key):
    """DRAM bytes (read + write) of one launch of the dominant kernel from the committed ncu --set full capture
    (profiles/ncu_traffic.json, written by tools/ncu_summarize.py from the .ncu-rep); None when there is no capture of the
    current kernel -- never a constant in this file."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p)).get(kernel_key)
        return (d["dram_bytes_per_launch"], d["note"]) if d else (None, "")
    except Exception:
        return None, ""


def randomise_bn(model, gen):
    """SURVEY 8d: make eval-mode BN non-trivial."""
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=gen) * 0.1)
                m.running_var.copy_(torch.rand(m.running_var.shape, generator=gen) + 0.5)
                m.weight.copy_(torch.rand(m.weight.shape, generator=gen) + 0.5)
                m.bias.copy_(torch.randn(m.bias.shape, generator=gen) * 0.1)


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons DURING the timed region (NVML, 20 Hz)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def usable_cpus():
    """Host threads this process can really use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per))))
    except Exception:
        pass
    return n


def cpu_port_time(n_frames, reps, threads):
    """Oracle leg (allowed to import oracle/): reference algorithm on the host cores."""
    import numpy as np
    from oracle import torch_port as TP
    from oracle.cases import cast_sd, fill_schema, smaat_unet_schema
    torch.set_num_threads(threads)
    sd = TP.to_torch_sd(cast_sd(fill_schema(smaat_unet_schema(C_IN, 1, 2), 0), np.float32))
    x = torch.rand(n_frames, C_IN, SIZE, SIZE)
    with torch.no_grad():
        TP.smaat_unet_forward(x[:1], sd)          # warm-up (oneDNN primitive creation)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            TP.smaat_unet_forward(x, sd)
            ts.append(time.perf_counter() - t0)
    return ts


def eager_gpu_baseline(model, xs, dev):
    """Reported-only: the reference's algorithm as eager PyTorch ops (ATen / cuDNN through oracle/torch_port.py) on the same
    GPU, same weights and B=32 input -- what a user of the unmodified reference gets on this box
    (train_precip_lightning.py:53-55), with cudnn.allow_tf32 False and True.  CUDA events, 3 warm-up + 5 timed forwards."""
    from oracle import torch_port as TP
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    out = {"unit": "frames/s", "batch": int(xs[0].shape[0]), "how": "oracle/torch_port.py on cuda (ATen/cuDNN eager, no graph), 3 warm-up + 5 timed"}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        for flag in (False, True):
            torch.backends.cudnn.allow_tf32 = flag
            torch.backends.cuda.matmul.allow_tf32 = flag
            with torch.no_grad():
                for i in range(3):
                    TP.smaat_unet_forward(xs[i % 2], sd)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for i in range(5):
                    TP.smaat_unet_forward(xs[i % 2], sd)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 5
            out["allow_tf32_true" if flag else "allow_tf32_false"] = {"value": xs[0].shape[0] / (ms * 1e-3), "ms_per_step": ms}
    except Exception as e:          # a reported-only leg must never take the bench line down
        out["error"] = repr(e)[:200]
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
        torch.cuda.empty_cache()
    return out


def train_leg(args, dev, rank, world, S, PAR, per_gpu_batches):
    """BASELINE configs[2] / configs[3]: the training step (forward + loss_func + metrics + backward + gradient all-reduce +
    Adam) through train.TrainSession, host batches copied in every step.  Reported per per-GPU batch size; with N > 1 also
    the all-reduce's own time (CUDA events around the NCCL calls), the step time with the collective switched off, and a
    replica-consistency check (post-reduce gradients identical on all ranks and equal to the mean of the pre-reduce ones)."""
    import torch.distributed as dist
    from smaat_unet_b200.train import TrainSession
    out = {"unit": "frames/s", "loss": "mse_loss(sum)/B, Adam(lr=1e-3) (regression_lightning.py:47-65)", "configs": []}
    if world > 1:
        out["nccl"] = {"nranks": dist.get_world_size(), "backend": dist.get_backend(), "version": ".".join(map(str, torch.cuda.nccl.version()))}
    for B in per_gpu_batches:
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        torch.manual_seed(0)
        model = S.SmaAt_UNet(C_IN, 1, kernels_per_layer=2).to(dev).train()
        try:
            sess = TrainSession(model, B, (C_IN, SIZE, SIZE), lr=1e-3, device=dev, use_graph=not args.no_graph)
        except torch.OutOfMemoryError:
            out["configs"].append({"batch_per_gpu": B, "error": "out of memory"})
            continue
        gen = torch.Generator().manual_seed(1 + rank)
        xs = [torch.rand((B, C_IN, SIZE, SIZE), generator=gen).pin_memory() for _ in range(2)]
        ys = [torch.rand((B, SIZE, SIZE), generator=gen).pin_memory() for _ in range(2)]

        def timed(k):
            for i in range(3):
                sess.step(xs[i % 2], ys[i % 2])
            PAR.barrier(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(k):
                sess.step(xs[i % 2], ys[i % 2])
            e1.record()
            PAR.barrier(dev)
            return PAR.reduce_max(e0.elapsed_time(e1), dev) / k

        k = max(5, min(args.steps, 10))
        ms = timed(k)
        cfg = {"batch_per_gpu": B, "global_batch": B * world, "ms_per_step": ms, "value": world * B / (ms * 1e-3),
               "launches_per_step": sess.launches_per_step, "two_phase_backward": sess._split is not None,
               "h2d_bytes_per_step": int(xs[0].numel() + ys[0].numel()) * 4, "max_mem_GB": torch.cuda.max_memory_allocated(dev) / 1e9}
        if world > 1:
            # --- replica consistency: identical parameters on all ranks after the timed steps
            cs = sess.replica_checksums()
            cfg["replicas_identical"] = all(c == cs[0] for c in cs)
            # --- the collective itself: pre-reduce gradients -> expected mean (separate all-reduce of a copy) vs the session's path
            sess.skip_allreduce = True
            sess.set_lr(0.0)
            sess.step(xs[0], ys[0])
            g_local = sess.flat_grad.clone()
            sess.skip_allreduce = False
            expect = g_local.clone()
            dist.all_reduce(expect, op=dist.ReduceOp.SUM)
            expect /= world
            sess.record_comm_timing = True
            sess.step(xs[0], ys[0])                       # same batch, lr = 0: same local gradients, now reduced by the session
            torch.cuda.synchronize(dev)
            got = sess.flat_grad
            scale = float(expect.abs().max())
            dev_err = float((got - expect).abs().max()) / max(scale, 1e-30)
            sums = torch.stack([got.double().sum(), got.double().abs().sum()])
            allsums = [torch.zeros_like(sums) for _ in range(world)]
            dist.all_gather(allsums, sums)
            cfg["allreduce_check"] = {"post_reduce_equals_mean_of_pre_reduce_rel_err": dev_err,
                                      "identical_on_all_ranks": all(torch.equal(a, allsums[0]) for a in allsums),
                                      "local_differs_from_mean": bool((g_local - expect).abs().max() > 0)}
            evs = sess.allreduce_events or []
            cfg["allreduce"] = [{"bytes": nb, "ms": e0.elapsed_time(e1)} for e0, e1, nb in evs]
            sess.record_comm_timing = False
            # --- step time with the collective switched off (replicas diverge: measurement only, last thing done)
            sess.set_lr(1e-3)
            sess.skip_allreduce = True
            ms_nc = timed(k)
            sess.skip_allreduce = False
            cfg["ms_per_step_without_allreduce"] = ms_nc
            cfg["exposed_allreduce_ms"] = ms - ms_nc
        out["configs"].append(cfg)
        sess.close()
        del sess
        if B == per_gpu_batches[0]:
            # memory/time trade-off (TrainSession(recompute_depthwise=True)): depthwise results recomputed in the backward
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats(dev)
            try:
                sess = TrainSession(model, B, (C_IN, SIZE, SIZE), lr=1e-3, device=dev, use_graph=not args.no_graph, recompute_depthwise=True)
                ms_r = timed(k)
                cfg["recompute_depthwise"] = {"ms_per_step": ms_r, "max_mem_GB": torch.cuda.max_memory_allocated(dev) / 1e9,
                                              "launches_per_step": sess.launches_per_step}
                sess.close()
                del sess
            except torch.OutOfMemoryError:
                cfg["recompute_depthwise"] = {"error": "out of memory"}
        del model, xs, ys
    torch.cuda.empty_cache()
    return out


def run_reference(args, rank):
    if rank != 0:
        return
    threads = usable_cpus()
    n = 4
    ts = cpu_port_time(n, args.warmup + args.steps, threads)[args.warmup:]
    sec = sum(ts)
    fps = n * len(ts) / sec
    sample = f"{len(ts)} steps x {n} frames of 12x{SIZE}x{SIZE} (B=32 workload, bounded), torch CPU fp32, {threads} threads"
    out = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sec / len(ts), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: full SmaAt-UNet forward, batch=32, 12->1ch 288x288 (bounded sample of 4 frames/step)",
                   "kernels_per_layer": 2, "eval": True},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default=os.environ.get("SMAAT_PW_MODE", "tf32x3"), choices=["tf32x3", "tf32", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-alt", action="store_true", help="skip the reported-only tf32 measurement")
    ap.add_argument("--no-train", action="store_true", help="skip the reported-only training-step leg")
    ap.add_argument("--leg-timeout", type=int, default=600, help="watchdog (s) over the explanatory legs after value / e2e are measured")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the output of the last timed step (rank 0's batch) to DIR/output.npy, float32; the inputs are "
                         "seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl b200")
    assert args.warmup >= 3 or args.impl == "reference", "timing rules: W >= 3"

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    nccl_log = None
    if world > 1 and "NCCL_DEBUG_FILE" not in os.environ:
        # keep NCCL's init lines (comm nranks, rings / NVLS) as evidence -- in a FILE (never stdout: the JSON line must stay alone
        # there), echoed to stderr by rank 0 at the end; the file goes to a temporary directory, never into the source tree
        try:
            nccl_log = os.path.join(tempfile.mkdtemp(prefix="smaat_bench_nccl_"), f"rank{rank}.log")
            os.environ["NCCL_DEBUG"] = "INFO"                 # (overrides a quieter preset: the file keeps stdout / stderr clean)
            os.environ["NCCL_DEBUG_SUBSYS"] = "INIT,ENV"
            os.environ["NCCL_DEBUG_FILE"] = nccl_log
        except OSError:
            nccl_log = None
    import torch.distributed as dist
    import smaat_unet_b200 as S
    from smaat_unet_b200 import parallel as PAR
    from smaat_unet_b200.engine import InferenceSession

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    PAR.init_from_env("nccl", dev)
    S.set_pointwise_mode(args.mode)

    gen = torch.Generator().manual_seed(0)
    torch.manual_seed(0)
    model = S.SmaAt_UNet(C_IN, 1, kernels_per_layer=2)
    randomise_bn(model, gen)
    model = model.to(dev).eval()
    note("building the inference session (warm-up + CUDA-graph capture)")
    sess = InferenceSession(model, B_PER_GPU, (C_IN, SIZE, SIZE), device=dev, use_graph=not args.no_graph)
    note("session ready")

    # two resident input batches (alternated); a step touches ~40 GB of activations >> 126 MB L2
    xs = [torch.rand((B_PER_GPU, C_IN, SIZE, SIZE), generator=gen).to(dev) for _ in range(2)]
    host = [torch.rand((B_PER_GPU, C_IN, SIZE, SIZE), generator=gen).pin_memory() for _ in range(2)]

    def barrier():
        PAR.barrier(dev)

    def reduce_max(v):
        return PAR.reduce_max(v, dev)

    def timed_replays(session):
        """W warm-up + K timed graph replays on alternating resident inputs; CUDA events, barrier + sync both sides, max over ranks."""
        for i in range(args.warmup):
            session.forward(xs[i % 2])
        barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for i in range(args.steps):
            session.forward(xs[i % 2])
        a1.record()
        barrier()
        return reduce_max(a0.elapsed_time(a1))

    # ---------------- device-resident throughput ("value") ----------------
    note("timing: device-resident replays")
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed_replays(sess)
    clocks = sampler.result()
    if args.dump_outputs and rank == 0:
        # the session's static output still holds the last timed replay's result (B=32 x 1 x 288 x 288, 10.6 MB)
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "output.npy"), sess.static_out.float().cpu().numpy())
    fps = world * B_PER_GPU * args.steps / (ms * 1e-3)
    launches = sess.launches_per_forward * args.steps        # C-ABI launches of one forward (counted at capture) x timed steps

    # ---------------- parity of the timed path, outside the timed region (rank 0) ----------------
    # two frames of the graph-replayed B=32 output vs the CPU restatement of the reference on the same input
    parity = None
    expect = [float(sess.forward(host[i].to(dev))[0, 0, 0, 0]) for i in range(2)]     # what e2e's checksum must add up to
    if rank == 0 and not args.no_cpu_baseline:
        import numpy as np
        from oracle import torch_port as TP
        sd_cpu = {k: v.detach().cpu() for k, v in model.state_dict().items()}
        fr = [3, 29]
        y_dev = sess.forward(xs[0])[fr].double().cpu().numpy()
        torch.set_num_threads(usable_cpus())
        with torch.no_grad():
            y_ref = TP.smaat_unet_forward(xs[0][fr].cpu(), sd_cpu).double().numpy()
        err = float(np.abs(y_dev - y_ref).max() / np.abs(y_ref).max())
        tol = {"tf32x3": 1e-4, "fp32": 1e-4, "tf32": 2e-2}[args.mode]
        parity = {"frames_checked": fr, "max_rel_err_vs_cpu_port": err, "tolerance": tol}
        assert err <= tol, f"bench: the timed path disagrees with the oracle: {err:.3e} > {tol:.1e}"

    # ---------------- end to end through the public API, host buffers ----------------
    note("timing: end to end (submit / collect)")
    for i in range(args.warmup):
        sess.submit(host[i % 2])
        sess.collect()
    barrier()
    t0 = time.perf_counter()
    chk = 0.0
    for i in range(args.steps):
        sess.submit(host[i % 2])
        if i >= 1:
            chk += float(sess.collect()[0, 0, 0, 0])       # read the result on the host
    chk += float(sess.collect()[0, 0, 0, 0])
    torch.cuda.synchronize()
    e2e_s = reduce_max(time.perf_counter() - t0)
    barrier()
    e2e_fps = world * B_PER_GPU * args.steps / e2e_s
    chk_expect = sum(expect[i % 2] for i in range(args.steps))
    assert abs(chk - chk_expect) <= 1e-6 * max(1.0, abs(chk_expect)), \
        f"bench: e2e results are not the results of the submitted batches (checksum {chk!r} != {chk_expect!r})"

    # ---------------- everything below is explanatory; the headline (value, e2e) is in hand.  A watchdog prints the line with what
    # has been measured so far if a later leg stalls (a reported-only leg must never cost the run its number) ----------------
    via_api = alt = gpu_eager = roof = roof_dw = roof_cbam = cpu = train = None
    kernels = {}
    e2e_meta = (sess.h2d_bytes_per_step, sess.d2h_bytes_per_step, sess.graph is not None)
    emitted = threading.Event()

    def build_out(incomplete=None):
        out = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "configs[1]: full SmaAt-UNet forward (eval), batch=32 per GPU, 12->1ch 288x288, kernels_per_layer=2",
                       "global_batch": B_PER_GPU * world, "pointwise": args.mode, "cuda_graph": e2e_meta[2],
                       "parallelism": f"batch-sharded x{world}, no collective",
                       "l2": "inputs alternate between 2 buffers; a step streams ~40 GB of activations (>> 126 MB L2)"},
            "roofline": roof, "depthwise_roofline": roof_dw, "cbam_roofline": roof_cbam, "kernels": kernels, "cpu_baseline": cpu,
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes_per_step": e2e_meta[0],
                    "d2h_bytes_per_step": e2e_meta[1], "ms_per_step": 1e3 * e2e_s / args.steps, "checksum": chk,
                    "checksum_expected": chk_expect},
            "parity": parity, "via_reference_api": via_api, "gpu_eager_baseline": gpu_eager, "train": train,
            "alt_mode": alt, "clocks": clocks, "gpu_launches": int(launches),
        }
        if incomplete:
            out["incomplete"] = incomplete
        return out

    def watchdog():
        if not emitted.wait(args.leg_timeout):
            if rank == 0:
                print(json.dumps(build_out(f"an explanatory leg did not finish within {args.leg_timeout} s; keys still null were not measured")),
                      flush=True)
            os._exit(0)

    threading.Thread(target=watchdog, daemon=True).start()

    # ---------------- the same forward through the plain reference-order calls only ----------------
    # (what a patch_reference() user of the unchanged reference classes executes: no OutConv-in-epilogue fusion)
    note("timing: plain reference-order calls")
    sess_api = InferenceSession(model, B_PER_GPU, (C_IN, SIZE, SIZE), device=dev, use_graph=not args.no_graph, serving_fusions=False)
    api_ms = timed_replays(sess_api)
    via_api = {"value": world * B_PER_GPU * args.steps / (api_ms * 1e-3), "unit": "frames/s", "ms_per_step": api_ms / args.steps,
               "gap_to_value": 1.0 - (ms / api_ms), "launches_per_step": sess_api.launches_per_forward,
               "note": "blocks called plainly in the reference's order (models/SmaAt_UNet.py:41-57); the CBAM->DownDS max-pool fusion is "
                       "reached through the plain calls, the OutConv epilogue fusion is not expressible there (standalone 1x1 kernel)"}
    del sess_api

    # ---------------- reported-only: same measurement in the single-pass TF32 mode ----------------
    # (what the reference itself computes on a GPU: cuDNN allow_tf32=True; ~1e-3 relative error instead of 1e-6)
    note("timing: tf32 mode / eager baseline / per-kernel roofline pass")
    if args.mode == "tf32x3" and not args.no_alt:
        S.set_pointwise_mode("tf32")
        sess2 = InferenceSession(model, B_PER_GPU, (C_IN, SIZE, SIZE), device=dev, use_graph=not args.no_graph)
        ams = timed_replays(sess2)
        alt = {"pointwise": "tf32", "value": world * B_PER_GPU * args.steps / (ams * 1e-3), "unit": "frames/s", "ms_per_step": ams / args.steps}
        del sess2
        S.set_pointwise_mode(args.mode)
        S.ops.bump_weights_generation()

    # ---------------- reported-only: eager PyTorch (ATen/cuDNN) on the SAME GPU -- the practical bar (SURVEY 2 / 8c) ----------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        gpu_eager = eager_gpu_baseline(model, xs, dev)

    # ---------------- roofline: per-kernel timing, CUDA events on the launching stream ----------------
    if rank == 0:
        hbm, tf32_peak, src = peaks()
        fwd = model.forward_serving
        with torch.no_grad():
            fwd(xs[0])
            torch.cuda.synchronize()
            with S.ops.profile() as prof:
                for i in range(3):
                    fwd(xs[i % 2])
            agg = prof.summary()
            # the last DS conv carries the fused OutConv epilogue (its own ABI entry): same kernel, count it with the others
            oc = agg.pop("smaat_dsconv_outconv_fwd", None)
            if oc is not None and "smaat_dsconv_fwd" in agg:
                for k_ in ("launches", "ms", "bytes", "flops"):
                    agg["smaat_dsconv_fwd"][k_] += oc[k_]
            elif oc is not None:
                agg["smaat_dsconv_fwd"] = oc
            if os.environ.get("SMAAT_BENCH_LAYERS"):
                for name, a in prof.summary(by_shape=True).items():
                    if "[" in name:
                        print(f"# {name:40s} {a['ms'] / 3:8.3f} ms  {a['bytes'] / a['ms'] / 1e6:7.0f} GB/s  {a['flops'] / a['ms'] / 1e9:7.1f} TF", file=sys.stderr)
        # tensor-core kernels issue 3 tf32 MMAs per product in tf32x3 mode (1 in tf32): issued flops = passes x algorithmic GEMM flops
        passes = {"tf32x3": 3.0, "tf32": 1.0, "fp32": 0.0}[args.mode]
        TENSOR = ("smaat_dsconv_fwd", "smaat_pw1x1_fwd")
        for name, a in agg.items():
            sec = a["ms"] * 1e-3
            gbs = a["bytes"] / sec / 1e9 if sec > 0 else 0.0
            tfl = a["flops"] / sec / 1e12 if sec > 0 else 0.0
            kernels[name] = {"launches_per_step": a["launches"] // 3, "ms_per_step": a["ms"] / 3, "algorithmic_GB_per_step": a["bytes"] / 3e9,
                             "achieved_GBps": gbs, "frac_hbm": gbs / hbm, "tflops": tfl}
            if name in TENSOR:
                kernels[name]["tf32_tflops_issued"] = passes * tfl
                kernels[name]["frac_tensor"] = passes * tfl / tf32_peak
        # dominant kernel of the measured path (by time): its own algorithmic bytes / its own time
        KNAMES = {"smaat_dsconv_fwd": "fused DS conv (depthwise 3x3 -> tcgen05 pointwise -> BN/ReLU, one kernel)",
                  "smaat_pw1x1_fwd": "pw1x1_tc_kernel", "smaat_dw3x3_fwd": "dw3x3_kernel"}
        dom = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
        d = kernels[dom]
        traffic, tnote = ncu_traffic(dom)
        f_h, f_t = d["frac_hbm"], d.get("frac_tensor", 0.0)
        # the bound is whichever floor is closer: both fractions are reported, `frac` is the one of the binding resource
        bound = "tensor" if f_t > f_h else "hbm"
        roof = {"kernel": KNAMES.get(dom, dom) + f" ({d['launches_per_step']} launches/step)", "bound": bound,
                "achieved": d["tf32_tflops_issued"] if bound == "tensor" else d["achieved_GBps"],
                "peak": tf32_peak if bound == "tensor" else hbm, "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
                "frac": f_t if bound == "tensor" else f_h, "frac_hbm": f_h, "frac_tensor": f_t, "peak_hbm_GBps": hbm,
                "peak_tf32_TFLOPs": tf32_peak, "peak_source": src, "traffic": traffic, "traffic_note": tnote,
                "algorithmic_bytes_per_step": d["algorithmic_GB_per_step"] * 1e9, "ms_per_step": d["ms_per_step"],
                "note": "frac_tensor counts ISSUED tf32 flops (3 MMA passes per product in tf32x3) against half the measured bf16 "
                        "cuBLAS peak; frac_hbm counts algorithmic bytes (input + output of the fused conv) against the measured copy bandwidth"}
        # CBAM at the level of the op (SURVEY 8d): all cbam_* launches of a forward against 3 |x| (the algorithmic minimum: the global
        # pools force a second read of x, plus one write) and against the 4 |x| the three-pass design moves
        ck = [k for k in kernels if k.startswith("smaat_cbam_")]
        if ck:
            t_c = sum(kernels[k]["ms_per_step"] for k in ck) * 1e-3
            x_bytes = 4.0 * B_PER_GPU * sum(c * (SIZE // d) ** 2 for c, d in ((64, 1), (128, 2), (256, 4), (512, 8), (512, 16)))
            roof_cbam = {"op": "CBAM x5 = ChannelAttention + SpatialAttention (models/layers.py:90-141), all smaat_cbam_* launches",
                         "launches_per_step": sum(kernels[k]["launches_per_step"] for k in ck), "ms_per_step": t_c * 1e3,
                         "x_bytes": x_bytes, "bound": "hbm", "peak": hbm, "unit": "GB/s", "peak_source": src,
                         "achieved_vs_3x_minimum": 3 * x_bytes / t_c / 1e9, "frac_vs_3x_minimum": 3 * x_bytes / t_c / 1e9 / hbm,
                         "achieved_4x_moved": 4 * x_bytes / t_c / 1e9, "frac_4x_moved": 4 * x_bytes / t_c / 1e9 / hbm,
                         "note": "per-kernel fractions (each kernel's own algorithmic bytes) are in `kernels`; the max-pool bytes written by "
                                 "the pool pass for DownDS are not counted here"}
        # the metric's named kernel -- "depthwise % HBM roofline": the standalone depthwise kernel over ALL 18 layers
        # (fusion switched off for this measurement pass only)
        S.set_fused_dsconv(False)
        with torch.no_grad():
            model(xs[0])
            torch.cuda.synchronize()
            with S.ops.profile() as prof2:
                for i in range(3):
                    model(xs[i % 2])
            a2 = prof2.summary().get("smaat_dw3x3_fwd")
        S.set_fused_dsconv(True)
        if a2:
            g2 = a2["bytes"] / (a2["ms"] * 1e-3) / 1e9
            t2, n2 = ncu_traffic("smaat_dw3x3_fwd")
            roof_dw = {"kernel": f"dw3x3_kernel ({a2['launches'] // 3} launches/step, all DS layers, unfused pass)", "bound": "hbm",
                       "achieved": g2, "peak": hbm, "unit": "GB/s", "frac": g2 / hbm, "peak_source": src,
                       "traffic": t2, "traffic_note": n2,
                       "algorithmic_bytes_per_step": a2["bytes"] / 3, "ms_per_step": a2["ms"] / 3}

    # ---------------- CPU baseline (oracle port), rank 0, N=1 only: the full B=32 batch, once ----------------
    note("cpu baseline")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = usable_cpus()
        n = B_PER_GPU
        ts = cpu_port_time(n, 1, threads)
        cpu = {"value": n / ts[0], "unit": "frames/s", "cores": threads, "kind": "port", "cpu_model": cpu_model_name(),
               "sample": f"1 timed forward of the full batch ({n} frames 12x{SIZE}x{SIZE}) after a 1-frame warm-up; oracle/torch_port.py "
                         f"(torch CPU fp32, {threads} threads)"}

    # ---------------- training step (configs[2]; configs[3] split when N > 1): reported beside the headline ----------------
    note("training leg")
    if not args.no_train:
        del sess
        S.ops.bump_weights_generation()
        batches = [B_PER_GPU] if world == 1 else sorted({B_PER_GPU, 256 // world})
        try:
            train = train_leg(args, dev, rank, world, S, PAR, batches)
        except Exception as e:          # a reported-only leg must never take the headline line down
            train = {"error": repr(e)[:300]}

    note("done")
    emitted.set()
    if rank == 0:
        out = build_out()
        print(json.dumps(out), flush=True)
        if nccl_log and os.path.exists(nccl_log):
            keep = [l.rstrip() for l in open(nccl_log, errors="replace") if any(k in l for k in ("nranks", "NVLS", "Connected all", "Channel 00/"))]
            for l in keep[:12]:
                print("[nccl] " + l[:220], file=sys.stderr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
