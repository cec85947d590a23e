#!/usr/bin/env python3
"""Headline benchmark: 20 ms-frame encode+decode throughput (frames/s) at 16 kHz.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm's CPU arm

One "step" = HOPS_PER_STEP (50) consecutive 20 ms hops = one second of audio of every stream, each hop PCM -> SoundStream
encoder -> RVQ -> packet bytes -> RVQ decode -> LyraGAN -> PCM, for `--streams` (default 4096) concurrent 16 kHz streams per GPU
(so `--steps 20` times 1000 hops: about a second of GPU time, enough for the clock sampler and for a stable wall-clock e2e).  One process per GPU (torchrun
for N > 1); streams are independent, so ranks shard them with no data-path collective (weak scaling); NCCL is
only used for the barrier and the max-over-ranks of the elapsed time.

The CPU arm (`--impl reference`, and the `cpu_baseline` object of the normal run) is the plain-C restatement
of the reference algorithm in oracle/ run on all host cores, one stream per thread like TFLite's
num_threads = 1 (the reference binary itself cannot be built offline: no bazel / TFLite / abseil, DESIGN.md).
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

METRIC = "20ms-frame encode+decode throughput (frames/s) @16kHz"
METRIC_PLC = "20ms-frame decode throughput with packet-loss concealment and noise tracking (frames/s) @16kHz"
UNIT = "frames/s"
SEED = 0x4C595241
HOPS_PER_STEP = 50          # one bench step = 50 hops = 1 s of audio per stream

# Algorithmic bytes per stream-frame (SURVEY.md §8d / BASELINE.md §2; fp32 state, read every state element once +
# write the new rows, + PCM + packet), split by the kernel that owns the state (DESIGN.md §4):
#   encoder: (13,808 + 6,128) * 4 = 79,744 B state + 640 B PCM + P B packet
#   decoder: (12,912 + 5,680) * 4 = 74,368 B state + 640 B PCM + P B packet
ALGO_BYTES = {
    "EncoderKernelA": (2032 + 2032) * 4 + 640,                 # first_layer + encoder_0 rings + simpleconv carry, PCM in
    "EncoderKernelB": (11776 + 4096) * 4,                      # the rest of the encoder state
    "RvqEncodeKernel": 0,                                      # + P (added per run)
    "RvqDecodeKernel": 0,                                      # + P
    "DecoderKernelC": (10880 + 3648) * 4,                      # bottleneck_2 .. decoder_1 state
    "DecoderKernelD": (2032 + 2032) * 4 + 640,                 # decoder_2 + last_layer state, PCM out
    "LogMelKernel": 640 + 2 * 640 + 160 * 4,                   # PCM in, carried hop read + written, 160 mel bins out
    "NoiseEstimatorKernel": 160 * 4 + 2 * 5 * 160 * 4 + 1,     # mel in, 5 x 160 floats of state read + written, flag out
}


def ncu_traffic(kernel, streams):
    """DRAM bytes per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(p) as f:
            d = json.load(f)
        if d.get("streams") == streams and kernel in d:
            return d[kernel]
    except (OSError, ValueError):
        pass
    return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clocks and clock-event (throttle) reasons while the timed region runs: NVML in-process every 20 ms
    (nvidia-ml-py), falling back to an `nvidia-smi -lms` subprocess when NVML cannot be loaded."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index, uuid=None):
        self.gpu = gpu_index
        self.uuid = uuid
        self.proc = None
        self.lines = []
        self.samples = []          # (sm_mhz, reasons bitmask)
        self.smax = None
        self.stop_flag = threading.Event()
        self.thread = None
        self.nvml = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByUUID(self.uuid.encode() if isinstance(self.uuid, str) else self.uuid) if self.uuid \
                else pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml

            def poll():
                while not self.stop_flag.is_set():
                    try:
                        self.samples.append((float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                             int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
                    except Exception:
                        pass
                    self.stop_flag.wait(0.02)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.thread.join(timeout=1.0)
            sm = [x[0] for x in self.samples]
            bits = 0
            for x in self.samples:
                bits |= x[1]
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.smax,
                    "reasons": sorted(v for k, v in self.REASONS.items() if bits & k), "samples": len(sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def host_cores():
    """CPU cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


def pin_rank_cores(local_rank, local_world):
    """Under torchrun every rank keeps its host threads (the synchronous calls' waiters) on its own slice of the allowed cores, so
    that the ranks of one box do not migrate onto each other's cores in the host-buffer pass.  Returns the slice size or None."""
    if local_world <= 1:
        return None
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // local_world
        if per < 2:
            return None
        os.sched_setaffinity(0, cores[local_rank * per:(local_rank + 1) * per])
        os.environ["LYRA_BENCH_PINNED"] = "1"      # host_cores() now reports this rank's slice
        return per
    except (AttributeError, OSError):
        return None


def host_pass_groups(requested, plc, ranks_sharing, cores, n):
    """Worker groups of the host-buffer pass.  requested > 0 wins; auto: 4 for the codec workloads when this rank has at least 16
    logical host cores for its 2 x 4 spin-waiting threads (hyper-thread siblings included - the configuration measured on one
    GPU), else 2 (the configuration measured under torchrun); the decoder-only workloads make short calls (0.1-0.4 ms of GPU
    work per hop) and do better with fewer, larger ones.  The result divides the stream count."""
    g = requested if requested > 0 else (4 if (not plc and ranks_sharing * 16 <= cores) else 2)
    g = max(1, g)
    while n % g:
        g -= 1
    return g


def host_pass_priorities(groups, bits, plc):
    """(encoder, decoder) stream priorities of the host-buffer pass; LYRA_BENCH_HOST_ENC_PRIORITY / ..._DEC_PRIORITY override.
    Equal by default (the synchronous calls of the 3.2 kbps workload lose 2-3 % with the encoder first, and four worker groups do
    well with equal priorities at every bit rate).  With only two worker groups the longer encoder chain of the higher bit rates
    (30 / 46 serial RVQ stages behind kernels A and B) holds the pipeline back and the encoder goes one step up: measured on one
    B200, 2 groups, 6.0 / 9.2 kbps: 5.60 / 5.53 M frames/s end to end against 5.06 / 4.80 M with equal priorities."""
    enc = -1 if (groups <= 2 and bits > 64 and not plc) else 0
    enc = int(os.environ.get("LYRA_BENCH_HOST_ENC_PRIORITY", str(enc)))
    dec = int(os.environ.get("LYRA_BENCH_HOST_DEC_PRIORITY", "0"))
    return enc, dec


def synth_pcm_np(n, nbuf, seed, kind="noise"):
    """Seeded synthetic input, `nbuf` distinct hops rotated through the steps (SURVEY.md section 8d):
    noise  — uniform noise at 0.25 full scale (the reference benchmark feeds uniform random audio, lyra/lyra_benchmark_lib.cc:233-239);
    speech — the reference's test clips tests/data/sample{1,2}_16kHz.wav tiled, stream i starting at offset (i * 7919) mod len."""
    import numpy as np
    if kind == "speech":
        import wave
        clips = []
        for name in ("sample1_16kHz.wav", "sample2_16kHz.wav"):
            with wave.open(os.path.join(ROOT, "tests", "data", name)) as w:
                clips.append(np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16))
        clip = np.concatenate(clips)
        start = (np.arange(n, dtype=np.int64) * 7919 + seed) % (len(clip) - 320 * nbuf)
        idx = start[None, :, None] + (np.arange(nbuf, dtype=np.int64) * 320)[:, None, None] + np.arange(320, dtype=np.int64)[None, None, :]
        return np.ascontiguousarray(clip[idx])
    rng = np.random.default_rng(seed)
    return rng.integers(-8192, 8192, size=(nbuf, n, 320), dtype=np.int16)


def run_cpu_arm(streams, frames, bits, threads):
    from oracle import oracle as O
    from lyra_b200 import _capi
    r = O.cpu_bench(_capi.MODEL_DIR, streams, frames, bits, threads, SEED)
    return r


def cpu_calibrated_sample(bits, threads, target_s):
    """Pick (streams, frames) so the CPU arm runs for about target_s seconds on `threads` cores."""
    probe = run_cpu_arm(threads, 4, bits, threads)
    per_frame_s = probe["wall_s"] / 4.0                       # one frame of every thread's stream
    frames = max(8, int(target_s / max(per_frame_s, 1e-6)))
    return threads, frames


def codec_workload(n, bits, world):
    return ("%d concurrent 16kHz streams per GPU, %.1f kbps encode+decode (BASELINE configs[%s]); one step = %d consecutive "
            "20 ms hops (1 s of audio per stream)" % (n, bits * 50 / 1000.0, "4" if world >= 8 else ("1" if n == 1024 else "2"), HOPS_PER_STEP))


def reference_arm(args, rank, world):
    """`--impl reference`: the reference algorithm's CPU implementation (oracle port) on all host cores."""
    if rank != 0:
        return 0
    threads = host_cores()
    bits = args.bits
    streams, frames = cpu_calibrated_sample(bits, threads, max(2.0, min(20.0, 120.0 / max(1, args.steps + args.warmup))))
    for _ in range(args.warmup):
        run_cpu_arm(streams, max(2, frames // 8), bits, threads)
    t_total, f_total, stage = 0.0, 0, [0.0] * 4
    for _ in range(args.steps):
        r = run_cpu_arm(streams, frames, bits, threads)
        t_total += r["wall_s"]
        f_total += r["frames"]
        stage = [a + b for a, b in zip(stage, r["stage_us"])]
    value = f_total / t_total
    sample = "%d streams x %d hops per step (one stream per thread), uniform noise 0.25 FS, %d bits" % (streams, frames, bits)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32+i8", "data": "synthetic",
        "config": {"workload": codec_workload(args.streams, bits, args.gpus),
                   "streams_per_gpu": args.streams, "bits_per_frame": bits, "hops_per_step": HOPS_PER_STEP,
                   "note": "CPU arm: bounded sample of the same workload; the reference binary cannot be built offline, "
                           "this is the oracle's C restatement of its algorithm (kind=port)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "stage_us_per_frame": {k: v / args.steps for k, v in zip(
                             ["feature_extractor", "quantizer_quantize", "quantizer_decode", "model_decode"], stage)}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)
    return 0


_JSON_FD = None


def protect_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL's version banner, for one) also print there, so the real
    stdout is set aside for the JSON line and file descriptor 1 is pointed at stderr for everything else."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


DUMP_MAX_BYTES = 63 * 10 ** 6      # --dump-outputs: all arrays together stay under 64 MB, .npy headers included


def write_outputs(out_dir, outputs):
    """--dump-outputs: every array (one row per stream) as float32 DIR/<name>.npy.  When they would exceed DUMP_MAX_BYTES
    together, every array keeps the same fixed, seeded sample of stream rows (in stream order).  Returns the rows kept."""
    import numpy as np
    n = len(next(iter(outputs.values())))
    row_bytes = sum(4 * (a.size // n) for a in outputs.values())
    rows = np.arange(n)
    if n * row_bytes > DUMP_MAX_BYTES:
        rows = np.sort(np.random.default_rng(SEED).choice(n, DUMP_MAX_BYTES // row_bytes, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a)[rows].astype(np.float32))
    return rows


def measure(args, n, bits, plc, loss, hops, warm_hops, kernel_hops, e2e_hops, world, rank, local_rank, decoder_mode, want_clocks,
            dump=False):
    """One configuration on this rank's GPU: device-resident throughput over `hops` hops, a serialised per-kernel pass, and the
    end-to-end pass through the host-buffer C ABI.  Returns a dict; multi-rank reductions (max over ranks) are done inside.
    dump: the result's "outputs" holds what each timed pass returned for the last hop it timed (decoded PCM, and the packets or,
    for the decoder-only workload, the comfort-noise flags), one row per stream."""
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from lyra_b200 import _capi

    P = (bits + 7) // 8
    # LyraEncoder and LyraDecoder are separate objects in the reference; here they are an encoder-only and a decoder-only
    # context with their own CUDA streams (and, in the host-buffer pass, their own host threads), so the encode of hop
    # i + 1 overlaps the decode of hop i on the GPU.  Every hop's decode consumes that hop's packets.
    enc = None if plc else _capi.Context(n, device=local_rank, roles="encoder")
    dec = _capi.Context(n, device=local_rank, roles="decoder")
    dec.set_decoder_mode(decoder_mode)
    ctxs = [c for c in (enc, dec) if c is not None]
    for c in ctxs:
        c.set_split(args.split)
    # Stream priorities (lyra_b200_set_priority, include/lyra_b200.h).  The device-resident pass queues many hops ahead through the
    # asynchronous *_device calls: there the encoder direction runs one step above the decoder (measured +2.8 % over equal
    # priorities, -3 % with the decoder first).  The host-buffer pass makes synchronous calls: equal priorities (measured: the
    # encoder-first setting costs it 2-3 %), so the encoder contexts go back to 0 before it.  Both settings are in `config`.
    prio_x = int(os.environ.get("LYRA_BENCH_DEVICE_ENC_PRIORITY", "-1"))
    prio_y = int(os.environ.get("LYRA_BENCH_DEVICE_DEC_PRIORITY", "0"))
    sx, sy = torch.cuda.Stream(priority=prio_x), torch.cuda.Stream(priority=prio_y)
    if enc:
        enc.set_priority(prio_x)             # its sub-batch streams
        enc.set_stream(sx.cuda_stream)
    dec.set_priority(prio_y)
    dec.set_stream(sy.cuda_stream)
    # worker groups: G context pairs of n / G streams each, used by the two timed passes; the full-size pair above serves the
    # per-kernel pass (one launch per kernel over all n streams)
    G = max(1, args.groups)
    while n % G:
        G -= 1
    ng = n // G
    if G == 1:
        groups = [(enc, dec, sx, sy)]
    else:
        groups = []
        for _ in range(G):
            e_ = None if plc else _capi.Context(ng, device=local_rank, roles="encoder")
            d_ = _capi.Context(ng, device=local_rank, roles="decoder")
            d_.set_decoder_mode(decoder_mode)
            gx, gy = torch.cuda.Stream(priority=prio_x), torch.cuda.Stream(priority=prio_y)
            d_.set_priority(prio_y)
            if e_:
                e_.set_priority(prio_x)
                e_.set_stream(gx.cuda_stream)
                e_.set_split(args.split)
            d_.set_stream(gy.cuda_stream)
            d_.set_split(args.split)
            groups.append((e_, d_, gx, gy))
    group_ctxs = [c for grp in groups for c in grp[:2] if c is not None]
    # the host-buffer pass has its own number of worker groups (--e2e-groups): synchronous calls need more call chains in flight to
    # cover their host turn-arounds and the serial RVQ stages than the asynchronous device pass does (measured at 6.0 / 9.2 kbps:
    # 4 groups 5.8 / 5.5 M frames/s end to end, 2 groups 5.1-5.5 / 4.7 M; the device pass is best at 2)
    ranks_sharing = 1 if os.environ.get("LYRA_BENCH_PINNED") else world
    Gh = host_pass_groups(args.e2e_groups, plc, ranks_sharing, host_cores(), n)
    # it runs 2 Gh waiting threads per rank: they sleep instead of spin when the box has fewer cores than that
    oversubscribed = args.host_wait == "sleep" or (args.host_wait == "auto" and
                                                   ranks_sharing * (2 * Gh + 1) > host_cores() * 3 // 4)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    NBUF = 8
    host = synth_pcm_np(n, NBUF, SEED + rank, args.input)
    d_pcm = [torch.from_numpy(host[i]).cuda() for i in range(NBUF)]
    d_pks = [torch.zeros((n, P), dtype=torch.uint8, device="cuda") for _ in range(NBUF)]
    d_out = torch.zeros((n, 320), dtype=torch.int16, device="cuda")
    ev_pk = [[torch.cuda.Event() for _ in range(NBUF)] for _ in range(max(G, 1) + 1)]      # [group][slot] packets written by the encoder
    ev_free = [[torch.cuda.Event() for _ in range(NBUF)] for _ in range(max(G, 1) + 1)]    # ... consumed by the decoder
    if plc:
        # packets of NBUF encoded hops + Bernoulli received masks (SURVEY.md section 8d config 4)
        tmp = _capi.Context(n, device=local_rank, roles="encoder")
        for i in range(NBUF):
            tmp.encode_device(n, d_pcm[i].data_ptr(), bits, d_pks[i].data_ptr())
        tmp.synchronize()
        tmp.close()
        mrng = np.random.default_rng(1234 + rank)
        h_masks = [(mrng.random(n) >= loss).astype(np.uint8) for _ in range(NBUF)]
        d_masks = [torch.from_numpy(m).cuda() for m in h_masks]
        d_flags = torch.zeros(n, dtype=torch.uint8, device="cuda")

    def run_device(first, count, grps, serial=False):
        """hops first .. first+count-1 over the given context groups (each group owns a contiguous slice of the streams);
        serial: hop i+1's encode waits for hop i's decode (per-kernel timing pass)"""
        m = n // len(grps)
        for i in range(first, first + count):
            b = i % NBUF
            for g, (e_, d_, gx, gy) in enumerate(grps):
                k = g if len(grps) > 1 else G        # event row: the full-size pair has its own
                off = g * m
                if plc:
                    d_.decode_plc_device(m, d_pks[b].data_ptr() + off * P, d_masks[b].data_ptr() + off, bits,
                                         d_out.data_ptr() + off * 640, d_flags.data_ptr() + off)
                    continue
                if serial and i > first:
                    gx.wait_event(ev_free[k][(i - 1) % NBUF])
                elif i - first >= NBUF:
                    gx.wait_event(ev_free[k][b])                   # the ring slot's previous packets have been decoded
                e_.encode_device(m, d_pcm[b].data_ptr() + off * 640, bits, d_pks[b].data_ptr() + off * P)
                ev_pk[k][b].record(gx)
                gy.wait_event(ev_pk[k][b])
                d_.decode_device(m, d_pks[b].data_ptr() + off * P, 0, bits, d_out.data_ptr() + off * 640)
                ev_free[k][b].record(gy)

    def drain(grps, onto):
        for _, _, gx, gy in grps:
            onto.wait_stream(gx)
            onto.wait_stream(gy)

    # ---------------- device-resident throughput (`value`) ----------------
    timer = torch.cuda.Stream()
    run_device(0, max(3, warm_hops), groups)
    barrier()
    launches0 = sum(c.launch_count for c in group_ctxs)
    sampler = None
    if want_clocks:
        try:
            gpu_uuid = "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
        except Exception:
            gpu_uuid = None
        sampler = ClockSampler(local_rank, gpu_uuid)
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(timer)
    for _, _, gx, gy in groups:          # nothing of the timed region starts before e0
        gx.wait_stream(timer)
        gy.wait_stream(timer)
    run_device(0, hops, groups)
    drain(groups, timer)
    e1.record(timer)
    torch.cuda.synchronize()
    elapsed_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    gpu_launches = sum(c.launch_count for c in group_ctxs) - launches0
    barrier()
    outputs = {}
    if dump:     # read before the per-kernel pass below reuses the buffers
        outputs["pcm"] = d_out.cpu().numpy()
        if plc:
            outputs["is_comfort_noise"] = d_flags.cpu().numpy()
        else:
            outputs["packets"] = d_pks[(hops - 1) % NBUF].cpu().numpy()
    # per-kernel roofline pass on the full-size context pair: the same hops with the kernels serialised (one launch per kernel
    # and hop over all n streams, no concurrent sub-batches, no encode/decode overlap), CUDA events around every launch
    full = [(enc, dec, sx, sy)]
    for c in ctxs:
        c.set_split(1)
    run_device(0, 3, full, serial=True)
    torch.cuda.synchronize()
    for c in ctxs:
        c.profile_enable(True)
    run_device(0, kernel_hops, full, serial=True)
    torch.cuda.synchronize()
    prof = {}
    for c in ctxs:
        for k, v in c.profile_read().items():
            if v[1]:
                prof[k] = v
        c.profile_enable(False)
    host_prio_x, host_prio_y = host_pass_priorities(Gh, bits, plc)
    if Gh == G:
        host_groups = groups
    else:
        if G > 1:
            for c in group_ctxs:
                c.close()
        host_groups = []
        for _ in range(Gh):
            e_ = None if plc else _capi.Context(n // Gh, device=local_rank, roles="encoder")
            d_ = _capi.Context(n // Gh, device=local_rank, roles="decoder")
            d_.set_decoder_mode(decoder_mode)
            host_groups.append((e_, d_, None, None))
    ng = n // Gh
    host_ctxs = [c for grp in host_groups for c in grp[:2] if c is not None]
    for e_, d_, _gx, _gy in host_groups:     # the host-buffer pass runs on the contexts' own streams, at its own priorities
        for c, prio in ((e_, host_prio_x), (d_, host_prio_y)):
            if c is not None:
                c.set_stream(None)
                c.set_priority(prio)
    for c in host_ctxs:
        c.set_blocking_sync(oversubscribed)
        c.set_split(args.e2e_split)
        c.set_graphs(args.graphs == "on")       # the dense host-buffer calls replay captured CUDA graphs (one per rotating buffer pair)
    barrier()
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    value = world * n * hops / (elapsed_ms / 1e3)

    # ---------------- end to end through the host-buffer C ABI (`e2e`) ----------------
    # pinned host buffers in, pinned host buffers out, every call synchronous (H2D, kernels, D2H inside it); the encoder and
    # the decoder are driven by one host thread each, the way a full-duplex server runs its uplink and downlink
    sys.setswitchinterval(5e-5)      # worker threads hand the GIL over quickly between their (GIL-free) C-ABI calls
    pin_in = [torch.from_numpy(host[i]).pin_memory() for i in range(NBUF)]
    pin_pks = [d_pks[i].cpu().pin_memory() for i in range(NBUF)]
    pin_out = torch.zeros((n, 320), dtype=torch.int16).pin_memory()
    lib = dec.api.lib
    errors = []
    if plc:
        pin_masks = [torch.from_numpy(h_masks[i]).pin_memory() for i in range(NBUF)]
        pin_flags = torch.zeros(n, dtype=torch.uint8).pin_memory()

    def ptr(tn, g, row_bytes):
        return C.c_void_p(tn.data_ptr() + g * ng * row_bytes)

    def run_host(count):
        threads = []
        for g, (e_, d_, _gx, _gy) in enumerate(host_groups):
            if plc:
                def downlink_only(g=g, d_=d_):
                    for i in range(count):
                        b = i % NBUF
                        if lib.lyra_b200_decode_plc(d_.h, None, ng, ptr(pin_pks[b], g, P), ptr(pin_masks[b], g, 1), bits,
                                                    ptr(pin_out, g, 640), ptr(pin_flags, g, 1)):
                            errors.append("decode: %s" % lib.lyra_b200_last_error(d_.h))
                threads.append(threading.Thread(target=downlink_only))
                continue
            ready, free = threading.Semaphore(0), threading.Semaphore(NBUF)

            def uplink(g=g, e_=e_, ready=ready, free=free):
                for i in range(count):
                    b = i % NBUF
                    free.acquire()
                    if lib.lyra_b200_encode(e_.h, None, ng, ptr(pin_in[b], g, 640), bits, ptr(pin_pks[b], g, P)):
                        errors.append("encode: %s" % lib.lyra_b200_last_error(e_.h))
                    ready.release()

            def downlink(g=g, d_=d_, ready=ready, free=free):
                for i in range(count):
                    b = i % NBUF
                    ready.acquire()
                    if lib.lyra_b200_decode(d_.h, None, ng, ptr(pin_pks[b], g, P), None, bits, ptr(pin_out, g, 640)):
                        errors.append("decode: %s" % lib.lyra_b200_last_error(d_.h))
                    free.release()

            threads += [threading.Thread(target=uplink), threading.Thread(target=downlink)]
        for x in threads:
            x.start()
        for x in threads:
            x.join()
        if errors:
            raise RuntimeError("host API failed: %s" % errors[0])

    run_host(NBUF + 1)               # warm-up: every rotating buffer pair has been through a call (graph captures included)
    barrier()
    t0 = time.perf_counter()
    run_host(e2e_hops)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * e2e_hops / float(t.item())
    if dump:
        outputs["e2e_pcm"] = pin_out.numpy().copy()
        if plc:
            outputs["e2e_is_comfort_noise"] = pin_flags.numpy().copy()
        else:
            outputs["e2e_packets"] = pin_pks[(e2e_hops - 1) % NBUF].numpy().copy()
    checksum = int(pin_out.to(torch.int64).sum().item())
    tile_streams = dec.tile_streams
    graph_replays = sum(c.graph_replays() for c in host_ctxs)
    for c in ctxs + (host_ctxs if Gh != G or G > 1 else []):
        c.close()
    return {"value": value, "elapsed_ms": elapsed_ms, "e2e_value": e2e_value, "e2e_s": float(t.item()), "prof": prof, "clocks": clocks,
            "gpu_launches": int(gpu_launches), "checksum": checksum, "G": G, "Gh": Gh, "oversubscribed": oversubscribed, "tile_streams": tile_streams, "stream_priority": {"device_pass": {"encoder": prio_x, "decoder": prio_y}, "host_pass": {"encoder": host_prio_x, "decoder": host_prio_y}},
            "P": P, "graph_replays": graph_replays, "outputs": outputs}


def roofline_of(res, n, bits, plc, world, hops, decoder_mode, clocks):
    """The `roofline` object of one measured configuration (per-kernel times from the serialised pass)."""
    peak, peak_src = measured_peaks()
    P = res["P"]
    kern = {}
    for k, (ms, cnt) in res["prof"].items():
        if cnt:
            ab = ALGO_BYTES.get(k, 0) + (P if k.startswith("Rvq") else 0)
            kern[k] = {"ms_per_launch": ms / cnt, "launches": cnt, "algo_bytes_per_launch": ab * n,
                       "achieved_gbs": ab * n / (ms / cnt * 1e-3) / 1e9}
    dom = max(kern, key=lambda k: kern[k]["ms_per_launch"])
    # decode_plc: decoder state traffic + PCM + packet + the estimator's state (5 x 160 floats read and written) and carried hop
    total_algo = (74368 + 640 + P + 1 + 2 * 5 * 160 * 4 + 2 * 640) if plc else (79744 + 640 + P) + (74368 + 640 + P)
    whole = total_algo * n * hops / (res["elapsed_ms"] / 1e3) / 1e9 if world == 1 else None
    roofline = {"bound": "hbm", "kernel": dom, "achieved": kern[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                "frac": kern[dom]["achieved_gbs"] / peak, "traffic": ncu_traffic(dom, n), "peak_source": peak_src,
                "kernel_share_of_step": kern[dom]["ms_per_launch"] / sum(v["ms_per_launch"] for v in kern.values()),
                "whole_step": {"algo_bytes_per_frame": total_algo, "achieved_gbs": whole, "frac": whole / peak if whole else None},
                "kernels": kern}
    if world == 1:
        # the CUDA-core roofline that binds the bit-exact layers (DESIGN.md section 5): ordered FFMA chains.  In the tensor decoder mode
        # only the encoder's fp32 layers and the decoder's bottleneck_2 stay on the FP32 pipe; the rest of the decoder's fp32 GEMMs run
        # on the tensor cores (kernel C: mma.sync TF32, kernel D: tcgen05 UMMA)
        enc_macs, dec_macs, dec_cuda_macs = 1475840, 1236736, 24576          # SURVEY.md section 8d, fp32 MACs per stream-frame
        fp32_macs = (0 if plc else enc_macs) + (dec_macs if decoder_mode == "exact" else dec_cuda_macs)
        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        pipe_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
        roofline["fp32_pipe"] = {"achieved": res["value"] * 2 * fp32_macs / 1e12, "peak": pipe_peak, "unit": "TFLOP/s",
                                 "frac": res["value"] * 2 * fp32_macs / 1e12 / pipe_peak, "fp32_macs_per_frame_on_cuda_cores": fp32_macs,
                                 "peak_source": "148 SMs x 128 FP32 lanes x 2 x SM clock sampled during the run"}
    return roofline


def main():
    global HOPS_PER_STEP
    protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps; one step = %d hops (1 s of audio) of every stream" % HOPS_PER_STEP)
    ap.add_argument("--warmup", type=int, default=3, help="untimed warm-up steps")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=4096, help="concurrent streams per GPU")
    ap.add_argument("--bits", type=int, default=None,
                    help="quantized bits per frame: 64 / 120 / 184 (3.2 / 6.0 / 9.2 kbps); default 64, and 120 at --gpus 8 (BASELINE configs[4])")
    ap.add_argument("--hops-per-step", type=int, default=HOPS_PER_STEP,
                    help="hops per bench step (default %d = 1 s of audio); profiling runs under ncu use 1" % HOPS_PER_STEP)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the short runs of the other BASELINE configs (other_configs)")
    ap.add_argument("--workload", default="codec", choices=["codec", "decode_plc"],
                    help="codec: encode+decode (the headline metric). decode_plc: BASELINE configs[3], decoder only with a received mask "
                         "through the reference's concealment / comfort-noise / fade state machine (lyra_b200_decode_plc)")
    ap.add_argument("--loss", type=float, default=0.1, help="decode_plc: packet loss probability (Bernoulli, seed 1234); 1.0 = all lost")
    ap.add_argument("--split", type=int, default=2, help="concurrent sub-batches of a dense call, device-resident pass (1..4)")
    ap.add_argument("--graphs", default="on", choices=["on", "off"], help="CUDA graphs for the host-buffer encode / decode calls of the e2e pass")
    ap.add_argument("--e2e-split", type=int, default=2, help="sub-batches in the host-buffer pass: their copies overlap the others' kernels")
    ap.add_argument("--e2e-groups", type=int, default=0, help="worker groups of the host-buffer (e2e) pass (0 = auto: 4, or 2 for the decoder-only workloads and on boxes with few host cores per rank); see --groups")
    ap.add_argument("--groups", type=int, default=2,
                    help="worker groups: the streams are divided among this many encoder/decoder context pairs, each pair with its own "
                         "CUDA streams and, in the host-buffer pass, its own two host threads (a server's worker threads); calls on "
                         "one context stay serialised")
    ap.add_argument("--input", default="noise", choices=["noise", "speech"],
                    help="synthetic input: uniform noise at 0.25 full scale (default) or the tiled reference speech clips")
    ap.add_argument("--host-wait", default="auto", choices=["auto", "spin", "sleep"],
                    help="how the worker threads of the host-buffer pass wait for the GPU (auto: sleep only when threads outnumber cores)")
    ap.add_argument("--decoder-mode", default="tensor", choices=["exact", "tensor"],
                    help="tensor (default): the decoder's fp32 GEMMs on the tensor cores (kernel D: tcgen05 UMMA), decoded PCM within "
                         "4 int16 LSB of the oracle, packets bit-exact; exact: decoded PCM bit-identical to the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed passes returned for their last hop as DIR/<name>.npy (float32, "
                         "one row per stream; pcm and packets, or is_comfort_noise for decode_plc; e2e_* from the host-buffer pass), "
                         "under 64 MB in all (a fixed, seeded sample of the streams when larger).  The inputs depend only on the "
                         "arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.bits is None:
        args.bits = 120 if args.gpus >= 8 else 64
    HOPS_PER_STEP = max(1, args.hops_per_step)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        return reference_arm(args, rank, world)

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    pinned = pin_rank_cores(local_rank, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # NCCL's version / debug lines must not land in front of the JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n, bits = args.streams, args.bits
    plc = args.workload == "decode_plc"
    hops = args.steps * HOPS_PER_STEP
    dump = args.dump_outputs is not None and rank == 0
    res = measure(args, n, bits, plc, args.loss, hops, max(3, args.warmup) * HOPS_PER_STEP, min(hops, 40), hops, world, rank, local_rank,
                  args.decoder_mode, want_clocks=True, dump=dump)
    value, e2e_value, clocks, P, G = res["value"], res["e2e_value"], res["clocks"], res["P"], res["G"]
    if dump:
        rows = write_outputs(args.dump_outputs, res["outputs"])
        print("bench.py: wrote %s (%d of %d streams) to %s" % (", ".join(sorted(res["outputs"])), len(rows), n, args.dump_outputs),
              file=sys.stderr)

    other = None
    if world == 1 and not args.no_other_configs and not plc:
        # short runs of the other BASELINE configs in the same process (value, e2e and the dominant kernel's roofline each)
        other = {}
        plan = [("configs[1]: 1024 streams, 3.2 kbps", 1024, 64, False, 0.0),
                ("configs[2]: 4096 streams, 6.0 kbps", 4096, 120, False, 0.0),
                ("configs[2]: 4096 streams, 9.2 kbps", 4096, 184, False, 0.0),
                ("configs[3]: 4096 streams, decoder only, concealment / comfort noise, loss 0.1", 4096, 64, True, 0.1),
                ("configs[3]: 4096 streams, decoder only, all packets lost (comfort noise)", 4096, 64, True, 1.0)]
        for name, on, obits, oplc, oloss in plan:
            if (on, obits, oplc) == (n, bits, plc):
                continue
            r = measure(args, on, obits, oplc, oloss, 150, 20, 10, 150, world, rank, local_rank, args.decoder_mode, want_clocks=False)
            rf = roofline_of(r, on, obits, oplc, world, 150, args.decoder_mode, clocks)
            other[name] = {"value": r["value"], "unit": UNIT, "hops_timed": 150, "ms_per_hop": r["elapsed_ms"] / 150,
                           "e2e": {"value": r["e2e_value"], "unit": UNIT},
                           "real_time_factor": r["value"] / (50.0 * on),
                           "roofline": {k: rf[k] for k in ("kernel", "achieved", "peak", "frac", "kernel_share_of_step")},
                           "kernel_ms": {k: v["ms_per_launch"] for k, v in rf["kernels"].items()}}

    if rank == 0:
        roofline = roofline_of(res, n, bits, plc, world, hops, args.decoder_mode, clocks)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads = host_cores()
            s, f = cpu_calibrated_sample(bits, threads, 12.0)
            r = run_cpu_arm(s, f, bits, threads)
            if plc:   # decoder stages only (dequantize + generative model), the part of the CPU port this workload runs
                r["frames_per_s"] = threads * 1e6 / (r["stage_us"][2] + r["stage_us"][3])
            cpu = {"value": r["frames_per_s"], "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": "%d streams x %d hops, one stream per thread, uniform noise 0.25 FS, %d bits" % (s, f, bits),
                   "note": "the oracle's op-by-op C interpreter of the reference graphs, not TFLite + XNNPACK (which cannot be built offline "
                           "and would be several times faster per core): a reported baseline, not a target",
                   "stage_us_per_frame": dict(zip(["feature_extractor", "quantizer_quantize", "quantizer_decode", "model_decode"], r["stage_us"]))}
        state_mb = n * EncDecStateBytes() / 1e6
        line = {
            "metric": METRIC_PLC if plc else METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": res["elapsed_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+i8 (decoder fp32 GEMMs: split tf32 on tensor cores)" if args.decoder_mode == "tensor" else "f32+i8",
            "data": "synthetic" if args.input == "noise" else "synthetic (reference speech clips tiled over the streams)",
            "config": {"workload": ("%d concurrent 16kHz streams per GPU, %.1f kbps, decoder only through the reference's packet-loss state machine "
                                    "(BASELINE configs[3]): received mask Bernoulli(%.2f, seed 1234), concealment -> fade -> comfort noise, "
                                    "log-mel + noise estimator on hops decoded from received packets; one step = %d hops (1 s of audio per stream)"
                                    % (n, bits * 50 / 1000.0, 1.0 - args.loss, HOPS_PER_STEP)) if plc else
                                   codec_workload(n, bits, world),
                       "streams_per_gpu": n, "bits_per_frame": bits, "hops_per_step": HOPS_PER_STEP, "tile_streams": res["tile_streams"],
                       "decoder_mode": args.decoder_mode, "sub_batches": {"device_pass": args.split, "host_pass": args.e2e_split}, "worker_groups": {"device_pass": G, "host_pass": res["Gh"]}, "stream_priority": res["stream_priority"],
                       "host_pass_cuda_graphs": {"enabled": args.graphs == "on", "replayed_calls": res.get("graph_replays", 0)},
                       "host_threads_wait": "sleep (blocking-sync event)" if res["oversubscribed"] else "spin",
                       "host_cores_per_rank": pinned if pinned else host_cores(),
                       "real_time_factor": value / (50.0 * n * world),
                       "l2": ("no flush needed: per-hop state working set %d x %.0f KB = %.0f MB exceeds the 126 MB L2; PCM inputs rotate over 8 buffers"
                              if state_mb > 126 else
                              "NOT flushed: the state working set %d x %.0f KB = %.0f MB fits in the 126 MB L2 at this stream count (as it would "
                              "in steady-state serving); PCM inputs rotate over 8 buffers; the headline configuration (4096 streams) exceeds L2")
                             % (n, EncDecStateBytes() / 1024.0, state_mb),
                       "parallelism": "streams sharded by rank, no data-path collective",
                       "execution": ("decoder context only" if plc else
                                     "full duplex: encoder-only and decoder-only context on their own CUDA streams (host-buffer pass: "
                                     "their own host threads); the encode of hop i+1 overlaps the decode of hop i, and every "
                                     "hop's decode consumes that hop's packets"),
                       "output_checksum": res["checksum"]},
            "e2e": {"value": e2e_value, "unit": UNIT, "seconds_timed": res["e2e_s"],
                    "h2d_bytes_per_step": HOPS_PER_STEP * (n * (P + 1) if plc else n * (640 + P)),
                    "d2h_bytes_per_step": HOPS_PER_STEP * (n * (640 + 1) if plc else n * (P + 640))},
            "gpu_launches": res["gpu_launches"],
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu,
        }
        if other is not None:
            line["other_configs"] = other
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


def EncDecStateBytes():
    # bytes of streaming state this implementation keeps per stream (fp32 rings + packed int8 rings), 4 kernels
    return 4 * (2032 + 6016 + 5888 + 2032)


if __name__ == "__main__":
    sys.exit(main())
