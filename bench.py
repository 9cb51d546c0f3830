#!/usr/bin/env python
"""bench.py — headline benchmark of the DSPi hot path on B200 (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One *step* = one pass of the 10-band EQ cascade over one batch: 65 536 channels x 6144 samples
(= 64 firmware packets of 96 frames @96 kHz) per GPU, channel-major float32, in place.
N>1 is launched by torchrun, one rank per GPU; channels shard with no data-path collective
(weak scaling: 65 536 channels per GPU, 524 288 at N=8 = BASELINE config 5).
Rank 0 prints ONE JSON line.

--dump-outputs DIR writes what the last timed step left in its buffer as DIR/eq_out.npy, so that two builds
can be compared output for output: the rows of a fixed, seeded sample of channels (every frame), float32, or
float64 for the int32 Q28 words (exact).  Inputs and parameters come from fixed seeds, so the same arguments
give the same inputs on every run.  With N>1 GPUs only rank 0 writes, so the sample is drawn from rank 0's channel
shard (the first channels of the job); the other shards are not in the file.
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "audio samples/sec (whole box) at 65536ch x 10-band EQ, 96 kHz; % HBM roofline"
CHANNELS_PER_GPU = 65536
FS = 96000.0
ALG_BYTES_PER_SAMPLE = 8          # 4 B read + 4 B written per channel-sample (SURVEY.md §8d)
DUMP_BYTES = 32 << 20             # --dump-outputs: size of the channel sample written


def dump_outputs(out_dir, buf, q28):
    """DIR/eq_out.npy: rows of ``buf`` (a [C][T] device tensor) for a sample of channels drawn with a fixed seed,
    as many as fit DUMP_BYTES (at least one)."""
    import torch
    Cn, T = buf.shape
    dtype = np.float64 if q28 else np.float32
    n = max(1, min(Cn, DUMP_BYTES // (T * np.dtype(dtype).itemsize)))
    rows = np.sort(np.random.default_rng(0).choice(Cn, n, replace=False))
    y = buf[torch.from_numpy(rows).to(buf.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "eq_out.npy"), y.astype(dtype))


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
                 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown",
                 0x100: "display_clock_setting"}
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nv:
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join()
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "n_samples": len(self.samples)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cpu_reference_run(variant, arith, frames, target_seconds, steps=1, warmup=0):
    """Times the reference's own dsp_process_channel_block (oracle/_ref, compiled from the unmodified
    sources) - or the oracle port when _ref is absent - on all host threads over a bounded sample of
    the same workload.  Returns (samples_per_s, info)."""
    from dspi_b200 import layouts as L, workloads as W
    from tests.orc import Oracle, Ref
    threads = host_threads()
    q = arith == "q28"
    use_ref = Ref.available()
    if use_ref:
        ref = Ref(arith)
        kind = "reference"
    else:
        ref = None
        kind = "port"
    orc = Oracle()
    # probe: 64 channels per thread, one packet row
    def make(Cn):
        params = W.eq_params_fast(variant if not q else "B", Cn, fs=FS, seed=1)
        bq = np.zeros(params.shape, L.BIQUAD_Q28 if q else L.BIQUAD_F32)
        orc.eq_coeffs(q, params, bq, FS)
        rng = np.random.default_rng(0)
        if q:
            x = rng.integers(-2**27, 2**27, (Cn, frames), dtype=np.int64).astype(np.int32)
        else:
            x = (rng.random((Cn, frames), dtype=np.float32) - np.float32(0.5))
        return bq, x

    def run(bq, x):
        if use_ref:
            return ref.eq_many_mt(bq, x, 10, 96, threads)
        return orc.eq_many_mt(arith, bq, x, 10, 96, threads)

    Cp = 16 * threads
    bq, x = make(Cp)
    dt = run(bq, x)
    rate = Cp * frames / dt
    Cn = int(max(threads, min(CHANNELS_PER_GPU, rate * target_seconds / frames)))
    Cn = max(threads, (Cn // threads) * threads)
    bq, x = make(Cn)
    for _ in range(warmup):
        run(bq.copy(), x.copy())
    times = []
    for _ in range(steps):
        times.append(run(bq, x))
    sps = Cn * frames * len(times) / sum(times)
    info = {"value": sps, "unit": "samples/s", "cores": threads, "kind": kind,
            "sample": f"{Cn} of {CHANNELS_PER_GPU} channels x {frames} samples, 96-sample packets, {len(times)} pass(es), "
                      f"{'oracle/_ref (reference sources, ' + ('-mfma -ffp-contract=fast' if arith == 'f32f' else '-ffp-contract=off' if arith == 'f32s' else '-fwrapv') + ')' if use_ref else 'oracle port'}",
            "seconds": sum(times)}
    return sps, info, Cn


def _time_eq(api, torch, arith, bq, Cn, T, steps=6, q=False):
    eng = api.EqEngine(arith, Cn)
    eng.upload(bq)
    bufs = []
    for i in range(3):
        if q:
            bufs.append(torch.randint(-2**27, 2**27, (Cn, T), dtype=torch.int32, device="cuda"))
        else:
            bufs.append(torch.rand((Cn, T), dtype=torch.float32, device="cuda") - 0.5)
    torch.cuda.synchronize()
    st = torch.cuda.ExternalStream(eng.stream)
    for i in range(3):
        eng.process_device(bufs[i % 3].data_ptr(), T, T)
    eng.sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(steps):
        eng.process_device(bufs[i % 3].data_ptr(), T, T)
    e1.record(st)
    eng.sync()
    ms = e0.elapsed_time(e1) / steps
    eng.close()
    del bufs
    torch.cuda.empty_cache()
    peak, _ = measured_peak_gbs()
    sps = Cn * T / (ms * 1e-3)
    return {"samples_per_s": sps, "ms_per_step": ms, "hbm_frac": sps * ALG_BYTES_PER_SAMPLE / 1e9 / peak, "channels": Cn, "frames": T}


def extra_configs(api, W, L, torch):
    """The other BASELINE configs, short runs (device-resident, CUDA events): reported beside the headline."""
    out = {}
    T = 6144
    try:
        p = W.eq_params_fast("B", CHANNELS_PER_GPU, fs=FS, seed=1)
        out["cfg2_variantB_f32_fused"] = _time_eq(api, torch, "f32f", api.compute_coefficients(p, fs=FS), CHANNELS_PER_GPU, T)
        p = W.eq_params_fast("A", CHANNELS_PER_GPU, fs=FS, seed=1)
        out["cfg2_variantA_f32_strict"] = _time_eq(api, torch, "f32s", api.compute_coefficients(p, fs=FS), CHANNELS_PER_GPU, T)
        p = W.eq_params_fast("B", 32768, fs=FS, seed=1)
        out["cfg4_q28_32768ch"] = _time_eq(api, torch, "q28", api.compute_coefficients(p, q28=True, fs=FS), 32768, T, q=True)
        # config 3: 8192 instances (65536 S/PDIF channels + 8192 PDM subs), s24 packets of 96 frames
        N, fpp, npk = 8192, 96, 64
        F = fpp * npk
        P, bq = W.chain_config3(N, fs=FS, seed=1)
        eng = api.ChainEngine("f32f", N, max_frames=F)
        eng.set_params(P)
        eng.upload_biquads(bq)
        pcm = torch.randint(0, 256, (N, F * 6), dtype=torch.uint8, device="cuda")
        spdif = torch.empty((N, 4, F, 2), dtype=torch.int32, device="cuda")
        pdm = torch.empty((N, F, 8), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        st = torch.cuda.ExternalStream(eng.stream)
        eng.process_device(pcm.data_ptr(), 24, npk, fpp, spdif.data_ptr(), pdm.data_ptr())
        eng.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record(st)
        for _ in range(reps):
            eng.process_device(pcm.data_ptr(), 24, npk, fpp, spdif.data_ptr(), pdm.data_ptr())
        e1.record(st)
        eng.sync()
        ms = e0.elapsed_time(e1) / reps
        part = eng.sm_partition()
        eng.close()
        out["cfg3_full_chain_8192inst"] = {"sm_partition": {"modulator": part[0], "other_stages": part[1]}, "instance_frames_per_s": N * F / (ms * 1e-3), "output_channel_samples_per_s": N * 9 * F / (ms * 1e-3),
                                           "ms_per_step": ms, "instances": N, "frames": F, "realtime_factor": (F / FS) / (ms * 1e-3),
                                           "bytes_per_instance_frame": {"pcm_in": 6, "spdif_out": 32, "pdm_out": 32}}
        # RP2040-shape Q28 chain: 8192 instances x (4 S/PDIF channels + 1 PDM sub)
        Pq, bqq_all = W.chain_config3_q28(N, fs=FS)
        engq = api.ChainEngineQ28(N, max_frames=F)
        engq.set_params(Pq)
        engq.upload_biquads(bqq_all)
        spq = torch.empty((N, 2, F, 2), dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        stq = torch.cuda.ExternalStream(engq.stream)
        engq.process_device(pcm.data_ptr(), 24, npk, fpp, spq.data_ptr(), pdm.data_ptr())
        engq.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stq)
        for _ in range(reps):
            engq.process_device(pcm.data_ptr(), 24, npk, fpp, spq.data_ptr(), pdm.data_ptr())
        e1.record(stq)
        engq.sync()
        msq = e0.elapsed_time(e1) / reps
        partq = engq.sm_partition()
        engq.close()
        out["cfg3_q28_chain_8192inst"] = {"instance_frames_per_s": N * F / (msq * 1e-3), "output_channel_samples_per_s": N * 5 * F / (msq * 1e-3),
                                          "ms_per_step": msq, "instances": N, "frames": F, "realtime_factor": (F / FS) / (msq * 1e-3), "sm_partition": {"modulator": partq[0], "other_stages": partq[1]}}
        # S/PDIF subframe encoder (the step after the chain): 32768 stereo streams x 6144 frames, 24 B per frame
        ns, Fs = 4 * N, 6144
        nrot = 3                                                            # rotate buffers: 1.6 GB + 3.2 GB each, larger than L2
        wbuf = [torch.randint(-2**23, 2**23, (ns, Fs, 2), dtype=torch.int32, device="cuda") for _ in range(nrot)]
        obuf = [torch.empty((ns, Fs, 2, 2), dtype=torch.int32, device="cuda") for _ in range(nrot)]
        torch.cuda.synchronize()
        cur = torch.cuda.current_stream()
        for i in range(3):
            api.spdif_encode_device(wbuf[i % nrot].data_ptr(), ns, Fs, obuf[i % nrot].data_ptr(), stream=cur.cuda_stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 9
        e0.record(cur)
        for i in range(reps):
            api.spdif_encode_device(wbuf[i % nrot].data_ptr(), ns, Fs, obuf[i % nrot].data_ptr(), stream=cur.cuda_stream)
        e1.record(cur)
        torch.cuda.synchronize()
        mss = e0.elapsed_time(e1) / reps
        peak, _ = measured_peak_gbs()
        gbs = ns * Fs * 24 / (mss * 1e-3) / 1e9
        out["spdif_encode_32768streams"] = {"frames_per_s": ns * Fs / (mss * 1e-3), "ms_per_step": mss, "streams": ns, "frames": Fs,
                                            "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                                                         "kernel": "spdif_encode_kernel", "algorithmic_bytes_per_launch": ns * Fs * 24}}
        del wbuf, obuf
    except Exception as e:                     # extras must never break the headline line
        out["error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="dspi_b200", choices=["dspi_b200", "reference"])
    ap.add_argument("--variant", default="A", choices=["A", "B"])
    ap.add_argument("--arith", default="f32f", choices=["f32f", "f32s", "q28"])
    ap.add_argument("--frames", type=int, default=6144)
    ap.add_argument("--channels", type=int, default=CHANNELS_PER_GPU)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output (a channel sample; with N>1 GPUs, of rank 0's shard only) to DIR/eq_out.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "dspi_b200":
        ap.error("--dump-outputs applies to the GPU path (--impl dspi_b200)")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    workload = (f"BASELINE configs[1]: {args.channels} channels x 10-band cascade @96 kHz, {args.arith}, variant "
                f"{args.variant} ({'all-TDF2 biquads' if args.variant == 'A' else '9 SVF + 1 TDF2'}), {args.frames} samples/step")

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        sps, info, Cn = cpu_reference_run(args.variant, args.arith, args.frames, target_seconds=4.0, steps=args.steps, warmup=args.warmup)
        line = {"metric": METRIC, "value": sps, "unit": "samples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * info["seconds"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"f32f": "f32", "f32s": "f32", "q28": "int32"}[args.arith], "data": "synthetic", "impl": "reference",
                "config": {"workload": workload, "sample_channels": Cn, "parallelism": f"{info['cores']} host threads"},
                "cpu_baseline": {k: info[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": sps, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import torch.distributed as dist
    from dspi_b200 import api, layouts as L, workloads as W

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    q = args.arith == "q28"
    Cn, T = args.channels, args.frames
    from dspi_b200 import sharding
    ch0, _ = sharding.shard_range(Cn * world, rank, world)    # contiguous channel shard of the whole job

    params = W.eq_params_fast(args.variant if not q else "B", Cn, fs=FS, seed=1, ch0=ch0)
    bq = api.compute_coefficients(params, q28=q, fs=FS)
    eng = api.EqEngine(args.arith, Cn, device=local_rank)
    eng.upload(bq)
    kernel_info = eng.kernel_info()       # float engines compile K1 for their topology vector here, outside the timed region

    # rotating input buffers, each larger than L2 (126 MB): 65536 x 6144 x 4 B = 1.5 GiB
    # inputs: the per-channel xorshift32 streams of SURVEY 8(d) (seed 123456789 ^ absolute channel), generated on the GPU
    nbuf = max(2, min(4, args.steps))
    bufs = W.inputs_device(Cn, T, nbuf, q, torch.device("cuda", local_rank), ch0=ch0)
    torch.cuda.synchronize()
    stream = torch.cuda.ExternalStream(eng.stream, device=torch.device("cuda", local_rank))

    def step(i):
        eng.process_device(bufs[i % nbuf].data_ptr(), T, T)

    for i in range(args.warmup):
        step(i)
    eng.sync()
    sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.start()
    ev0.record(stream)
    for i in range(args.steps):
        step(i)
    ev1.record(stream)
    eng.sync()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, bufs[(args.steps - 1) % nbuf], q)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    total_samples = float(Cn) * T * args.steps * world
    value = total_samples / (ms * 1e-3)

    # per-kernel roofline: the step IS one launch of the cascade kernel
    peak, peak_src = measured_peak_gbs()
    per_gpu_sps = float(Cn) * T * args.steps / (ms * 1e-3)
    achieved = per_gpu_sps * ALG_BYTES_PER_SAMPLE / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "peak_source": peak_src, "kernel": "eq_q28_kernel" if q else ("eq_f32_jit" if kernel_info.startswith("jit") else "eq_f32_kernel"),
                "kernel_variant": kernel_info,
                "algorithmic_bytes_per_launch": Cn * T * ALG_BYTES_PER_SAMPLE,
                "note": ("integer-multiply bound, not HBM bound: 15 IMAD per band-sample on the half-rate IMAD pipe (DESIGN.md K2)" if q else
                         "FP32-issue bound, not HBM bound: see DESIGN.md (60 FMA-pipe lane-ops per sample)")}
    tr = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr):
        try:
            roofline["traffic"] = json.load(open(tr)).get(f"{roofline['kernel']}:{args.arith}:{args.variant}")
        except Exception:
            pass

    # end to end through the C ABI with HOST buffers (pinned): H2D + kernel(s) + D2H inside the timed region
    e2e = None
    if not args.no_e2e:
        numa_node = api.bind_host_to_device(local_rank)   # staging memory local to this GPU's PCIe root (before it is allocated)
        pin = api.PinnedBuffer((Cn, T), np.int32 if q else np.float32)
        src = bufs[0].cpu().numpy()
        pin.array[...] = src
        n_e2e = max(2, min(5, args.steps))
        eng.process_host(pin.array)                       # warm-up (allocates staging)
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            eng.process_host(pin.array)
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        e2e = {"value": float(Cn) * T * n_e2e * world / dt, "unit": "samples/s", "h2d_bytes_per_step": Cn * T * 4 * world,
               "d2h_bytes_per_step": Cn * T * 4 * world, "steps": n_e2e, "numa_node": numa_node,
               "path": "dspi_eq_process_host: pinned host [C][T] -> channel-chunked cudaMemcpyAsync H2D / kernel / D2H: copy-in stream, copy-out stream, a kernel stream per staging buffer (48 MiB chunks, ring of 8)"}
        pin.free()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        _, cpu, _ = cpu_reference_run(args.variant, args.arith, T, target_seconds=10.0)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # ---- N>1: frames originate on rank 0 and travel over NCCL/NVLink (scatter in, gather out) ----
    nccl = None
    if world > 1:
        total = Cn * world
        full = None
        if rank == 0:
            full = torch.rand((total, T), dtype=torch.float32, device="cuda") - 0.5 if not q else \
                torch.randint(-2**27, 2**27, (total, T), dtype=torch.int32, device="cuda")
        dt_t = torch.int32 if q else torch.float32
        sg = sharding.native_scatter_gather(eng, local_rank)       # dspi_sg_*: NCCL send / recv issued from the C library

        def sg_step():
            sg.process(full.data_ptr() if rank == 0 else 0, total, T, 0)      # 0: chunk count chosen by the library
        sg_step()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        n_sg = 3
        for _ in range(n_sg):
            sg_step()
        torch.cuda.synchronize()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        nccl = {"value": float(total) * T * n_sg / float(dt.item()), "unit": "samples/s", "steps": n_sg,
                "path": "rank 0 holds all frames: dspi_sg_process - row chunks (count chosen from transfer / kernel time), one NCCL group per step carries chunk j out and chunk j-L back while the kernels work on the chunks in between, each on its own stream (L from kernel / step time)",
                "bytes_over_nvlink_per_step": int(total - Cn) * T * 4 * 2}
        del full
        sg.close()

    other = None
    if rank == 0 and world == 1 and not args.no_extras:
        other = extra_configs(api, W, L, torch)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": {"f32f": "f32", "f32s": "f32", "q28": "int32"}[args.arith], "data": "synthetic",
                "config": {"workload": workload, "channels_per_gpu": Cn, "frames_per_step": T, "sample_rate_hz": FS,
                           "arith": args.arith, "variant": args.variant, "parallelism": f"channel-sharded dp{world}, no collective on the data path",
                           "l2": f"inputs larger than L2: {nbuf} rotating buffers of {Cn * T * 4 / 2**30:.2f} GiB", "inputs": "per-channel xorshift32 streams (seed 123456789 ^ channel), s16 / 65536", "layout": "channel-major [C][T], in place"},
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
                "nccl_scatter_gather": nccl, "other_configs": other,
                "realtime_factor": value / (Cn * world * FS)}
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
