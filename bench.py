#!/usr/bin/env python3
"""bench.py -- SOLO encode+decode packets/s on B200 (BASELINE.json metric), contract of the build brief.

A "step" is one packet wave: every resident stream encodes one 40 ms / 16 kHz packet and decodes it again
(lostflag 4).  Workload = BASELINE.json configs[2]: 65 536 concurrent streams per GPU, speech-replay input
(SURVEY.md 8(d) synthetic batch (i)), encoder rate 13 600 b/s.  Weak scaling: every rank owns 65 536 streams
(configs[3] = 8 x 65 536); streams never interact, so there is no data-path collective.

  value : packets/s with PCM already resident in HBM (device entry points of the C ABI, CUDA events, max over ranks)
  e2e   : packets/s through the host entry points of the C ABI (pinned host buffers; H2D of the PCM, D2H of the
          payloads, H2D of payloads/flags and D2H of the decoded PCM are all inside the timed region)
  roofline     : encode kernel (dominant), algorithmic bytes / CUDA-event kernel time vs measured HBM copy peak
  cpu_baseline : the unmodified reference (oracle/_ref: FIX encoder + FLP decoder) on all host cores, bounded sample

`--impl reference` times only that CPU baseline and prints the same JSON shape.
`--dump-outputs DIR` also writes what the last timed step of both paths returned, for a fixed sample of the streams
(see dump_outputs), so that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "40ms 16kHz frames enc+dec/sec at batch=65536; concurrent real-time streams"
UNIT = "packets/s"
CAP = 128           # bytes per payload row (max observed 117 at 13.6 kb/s; the kernel honours the cap like bits_write)
RATE = 13600
MEAN_PAYLOAD = 83.0  # refined with the measured mean below


def load_clip():
    return np.load(os.path.join(ROOT, "tests", "golden", "speech_clip.npz"))["pcm"]


def speech_replay(clip, stream_ids, n_packets):
    n = len(clip)
    s = np.asarray(stream_ids, dtype=np.int64)
    off = (s * 7919 * 640) % n
    idx = np.arange(640, dtype=np.int64)
    sh = (s & 3).astype(np.int16)
    out = np.empty((n_packets, len(s), 640), np.int16)
    for p in range(n_packets):
        ii = (off[:, None] + p * 640 + idx[None, :]) % n
        out[p] = clip[ii] >> sh[:, None]
    return out


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_summary():
    """profiles/ncu_summary.json (tools/profile_round.py): per kernel the DRAM bytes, issue-slot utilisation and warp
    instructions of one `ncu --set full` launch.  bench.py never runs under a profiler; these are the committed captures."""
    p = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        d = json.load(open(p))
        return d if "kernels" in d else None
    except Exception:
        return None


def ncu_traffic(kernel, streams_per_launch):
    """DRAM bytes (read + write) of `kernel` per launch, scaled from the capture's streams per launch to this run's."""
    d = ncu_summary()
    try:
        k = d["kernels"][kernel]
        return k["dram_bytes_per_launch"] / k["streams_per_launch"] * streams_per_launch
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons while the timed region runs (B200_PROFILING.md clocks line)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=5)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for nme, v in zip(names, r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores():
    """Cores this process may actually use: the affinity mask, capped by the cgroup CPU quota (a container that sees 128
    CPUs but is throttled to a few would otherwise run the baseline 10x oversubscribed -- round 1's 5x spread between hosts)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
            break
        except Exception:
            continue
    if quota:
        n = max(1, min(n, int(quota)))
    return min(n, 256)


# CPU baseline sample: one pinned thread per usable core, 8 streams x 250 packets = 2 000 timed packets per thread
CPU_SPT, CPU_PK = 8, 250


def run_cpu_baseline(threads, streams_per_thread, packets):
    """Unmodified reference on the host cores: oracle/_ref/cpu_baseline (built by `make -C oracle`)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "cpu_baseline")
    libdir = os.path.join(ROOT, "oracle", "_ref")
    if not (os.path.exists(exe) and os.path.exists(os.path.join(libdir, "libjc1_fix.so"))):
        return None
    with tempfile.NamedTemporaryFile(suffix=".pcm", delete=False) as f:
        load_clip().tofile(f)
        path = f.name
    try:
        out = subprocess.run([exe, libdir, path, str(threads), str(streams_per_thread), str(packets), str(RATE), "1"],
                             capture_output=True, text=True, timeout=600).stdout.strip().splitlines()[-1]
        return json.loads(out)
    finally:
        os.unlink(path)


def bench_reference(args, rank):
    if rank != 0:
        return
    cores = usable_cores()
    vals = []
    spt, pk = CPU_SPT, CPU_PK
    t0 = time.time()
    res = None
    for i in range(args.warmup + args.steps):
        res = run_cpu_baseline(cores, spt, pk)
        if res is None:
            emit({"impl": "reference", "unavailable": "oracle/_ref not built (run make -C oracle in the build container)"})
            return
        if i >= args.warmup:
            vals.append(res["packets_per_s"])
    v = float(np.mean(vals))
    sample = "%d pinned threads (one per usable core; %d CPUs visible) x %d streams x %d packets per step, speech-replay input, rate %d" % (cores, os.cpu_count() or 0, spt, pk, RATE)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * cores * spt * pk / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32/int16 fixed point (encoder), f32 (decoder high band)", "data": "synthetic (speech-replay of the codec's test clip)",
        "config": {"workload": "configs[2]: enc+dec round trip, speech-replay, 13.6 kb/s (bounded CPU sample)", "streams": cores * spt},
        "streams_rt": v / 25.0,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample,
                         "packets_per_s_per_core": v / cores, "cpus_visible": os.cpu_count()},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "wall_s": time.time() - t0,
    }
    emit(line)


def measure_root_ingest(args, dist, solo_b200, torch, rank, world, local_rank, dev, N, K, W, T, d_pcm, d_flags, d_ret, d_out, d_nb, stream, value):
    """configs[3] as BASELINE words it: one ingest point.  Rank 0 owns the PCM of ALL streams and receives all payloads / decoded
    PCM in its HBM; the other ranks map those buffers (CUDA IPC, solo_b200/shard.py) and hand their rows to the same *_device
    entry points: the band-split kernel pulls PCM over NVLink / NVSwitch, the entropy-coding and synthesis kernels push their rows
    back -- scatter and gather are fused into the kernels that consume / produce the data, no NCCL transfer step, no staging copy."""
    from solo_b200.shard import share_from_root
    lo = rank * N

    def agree(ok):      # every rank takes part, so that a failure on one rank ends the measurement on all of them together
        f = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        return bool(f.item())

    err = None
    r_pcm = r_bits = r_nb = r_out = None
    if rank == 0:
        try:
            r_pcm = torch.empty((T, world * N, 640), dtype=torch.int16, device=dev)
            r_bits = torch.zeros((world * N, CAP), dtype=torch.uint8, device=dev)
            r_nb = torch.zeros((world * N, 2), dtype=torch.int16, device=dev)
            r_out = torch.zeros((world * N, 640), dtype=torch.int16, device=dev)
        except Exception as ex:
            err = ex
    if not agree(err is None):
        return {"error": "root buffers: %s" % (str(err)[:160] if err else "failed on rank 0")}
    try:
        r_pcm, r_bits, r_nb, r_out = (share_from_root(t_) for t_ in (r_pcm, r_bits, r_nb, r_out))
        r_pcm[:, lo:lo + N].copy_(d_pcm)             # setup (untimed): every rank deposits its input rows at the root
        torch.cuda.synchronize()
    except Exception as ex:
        err = ex
    if not agree(err is None):
        return {"error": "peer mapping: %s" % (str(err)[:160] if err else "failed on another rank")}
    dist.barrier()
    enc_r = solo_b200.EncoderBatch(N, rate=RATE, device=local_rank)
    dec_r = solo_b200.DecoderBatch(N, device=local_rank)
    pb, pn, po = r_bits[lo:lo + N].data_ptr(), r_nb[lo:lo + N].data_ptr(), r_out[lo:lo + N].data_ptr()

    def step_root(t):
        enc_r.encode_device(r_pcm[t, lo:lo + N].data_ptr(), pb, CAP, pn, stream)
        dec_r.decode_device(po, pb, CAP, pn, d_flags.data_ptr(), d_ret.data_ptr(), stream)

    for t in range(W):
        step_root(t)
    torch.cuda.synchronize()
    dist.barrier()
    e0r, e1r = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0r.record()
    for t in range(W, T):
        step_root(t)
    e1r.record()
    torch.cuda.synchronize()
    t_ = torch.tensor([e0r.elapsed_time(e1r)], device=dev)
    dist.all_reduce(t_, op=dist.ReduceOp.MAX)
    root_ms = float(t_.item())
    dist.barrier()
    same = bool(torch.equal(r_out[lo:lo + N], d_out)) and bool(torch.equal(r_nb[lo:lo + N], d_nb))   # same streams, same packets
    root = {"value": world * N * K / (root_ms / 1e3), "unit": UNIT, "ms_per_step": root_ms / K,
            "vs_rank_ingest": (world * N * K / (root_ms / 1e3)) / value,
            "nvlink_bytes_per_step": (world - 1) * N * (1280 + 2 * (CAP + 4) + 1280),
            "identical_to_rank_ingest": same,
            "how": "rank 0 holds PCM in / payloads + PCM out of all %d streams; peers read / write them inside the codec kernels over NVLink (CUDA IPC mapping), max over ranks" % (world * N)}
    enc_r.close(); dec_r.close()
    del r_pcm, r_bits, r_nb, r_out, pb, pn, po
    dist.barrier()
    return root


def bind_to_gpu_numa(index):
    """Run this rank (and first-touch its pinned host buffers) on the CPUs next to its GPU: NVML's CPU affinity of the device,
    intersected with what the process may use.  Returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 64
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (int(v) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return "%d CPUs of the GPU's NUMA node (%d..%d)" % (len(cpus), min(cpus), max(cpus))
    except Exception as ex:
        return "not bound (%s)" % type(ex).__name__
    return "not bound"


DUMP_STREAMS = 8192   # 2 paths x 8192 streams x (128 + 2 + 640 + 1) float32 values = 51 MB


def dump_outputs(out_dir, torch, n_streams, paths):
    """Write the last timed step's outputs of each path as <path>_<name>.npy (float32), rows of a fixed seeded sample of
    the streams (stream_index.npy, float64).  Payload bytes past the payload's length are not part of the result and
    are written as 0."""
    os.makedirs(out_dir, exist_ok=True)
    rows = np.sort(np.random.default_rng(0).choice(n_streams, min(n_streams, DUMP_STREAMS), replace=False))
    np.save(os.path.join(out_dir, "stream_index.npy"), rows.astype(np.float64))
    for path, arrays in paths.items():
        got = {k: t.index_select(0, torch.as_tensor(rows, device=t.device)).cpu().numpy() for k, t in arrays.items()}
        got["payload"][np.arange(CAP)[None, :] >= got["nbytes"][:, :1]] = 0
        for k, a in got.items():
            np.save(os.path.join(out_dir, "%s_%s.npy" % (path, k)), a.astype(np.float32))


def emit(line):
    """The one JSON line goes to the process's original stdout; everything else that libraries print to file descriptor 1
    (NCCL's version banner, for instance) was redirected to stderr at start-up."""
    OUT.write(json.dumps(line) + "\n")
    OUT.flush()


OUT = sys.stdout


def main():
    global OUT
    OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="solo_b200", choices=["solo_b200", "reference"])
    ap.add_argument("--streams", type=int, default=65536, help="streams per GPU")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-root-ingest", action="store_true", help="skip the single-ingest-point measurement (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0's streams) to DIR")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "solo_b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        bench_reference(args, rank)
        return

    import torch
    import solo_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- libsolo_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    N = args.streams
    K, W = args.steps, args.warmup
    T = K + W
    clip = load_clip()
    sids = np.arange(rank * N, (rank + 1) * N)
    dev = torch.device("cuda", local_rank)

    enc = solo_b200.EncoderBatch(N, rate=RATE, device=local_rank)
    dec = solo_b200.DecoderBatch(N, device=local_rank)

    # ---------------- device-resident throughput (`value`) ----------------
    # Each step consumes a different 84 MB PCM wave (inputs + 0.9 GB of codec state >> 126 MB L2: no L2 flush needed).
    host_pcm = torch.from_numpy(speech_replay(clip, sids, T)).pin_memory()      # [T, N, 640] int16
    d_pcm = host_pcm.to(dev, non_blocking=True)
    # Encoder wave then decoder wave on one CUDA stream.  (Running the two batch objects on separate streams so that
    # decode(t) overlaps encode(t+1) gains nothing -- tools/overlap_check.py, 25.6 vs 25.8 ms: a later grid's blocks are only
    # placed once the earlier grid has none left, so the kernels overlap at their tails -- DESIGN.md section 6.)
    d_bits = torch.zeros((N, CAP), dtype=torch.uint8, device=dev)
    d_nb = torch.zeros((N, 2), dtype=torch.int16, device=dev)
    d_flags = torch.full((N,), 4, dtype=torch.int32, device=dev)
    d_out = torch.zeros((N, 640), dtype=torch.int16, device=dev)
    d_ret = torch.zeros((N,), dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device(t):
        enc.encode_device(d_pcm[t].data_ptr(), d_bits.data_ptr(), CAP, d_nb.data_ptr(), stream)
        dec.decode_device(d_out.data_ptr(), d_bits.data_ptr(), CAP, d_nb.data_ptr(), d_flags.data_ptr(), d_ret.data_ptr(), stream)

    for t in range(W):
        step_device(t)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    solo_b200.profile_enable(True)
    l0 = solo_b200.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for t in range(W, T):
        step_device(t)
    e1.record()
    torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1)
    launches = solo_b200.kernel_launches() - l0
    prof = solo_b200.profile_read()
    solo_b200.profile_enable(False)
    mean_payload = float(d_nb[:, 0].float().mean().item())
    ret_ok = bool((d_ret == 0).all().item())
    if dist:
        t_ = torch.tensor([dev_ms], device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        dev_ms = float(t_.item())
    value = world * N * K / (dev_ms / 1e3)

    # ---------------- configs[3] as BASELINE words it: one ingest point (`root_ingest`, N > 1 only) ----------------
    # Rank 0 owns the PCM of ALL streams and receives all payloads / decoded PCM in its HBM; the other ranks map those buffers
    # (CUDA IPC, solo_b200/shard.py) and hand their rows to the same *_device entry points: the band-split kernel pulls PCM
    # over NVLink / NVSwitch, the entropy-coding and decoder kernels push their rows back -- scatter and gather are fused into
    # the kernels that consume / produce the data, no NCCL transfer step and no staging copy.
    root = None
    if dist and not args.no_root_ingest:
        try:
            root = measure_root_ingest(args, dist, solo_b200, torch, rank, world, local_rank, dev, N, K, W, T, d_pcm, d_flags, d_ret, d_out, d_nb, stream, value)
        except Exception as ex:      # the per-rank numbers above stand on their own
            root = {"error": "%s: %s" % (type(ex).__name__, str(ex)[:200])}
        dist.barrier()

    # ---------------- end-to-end through the host entry points (`e2e`) ----------------
    # fresh codec objects are not needed: the streams simply continue with the next packets of the same input
    # Public host API (solo_b200_enc_batch_encode_host / solo_b200_dec_batch_decode_host): every call copies its step's
    # inputs from pinned host memory, runs the kernels, and copies the results back before it returns (inside the call
    # the wave is pipelined in chunks, so most of the copy time hides behind the kernels of the neighbouring chunk).
    h_bits = torch.zeros((N, CAP), dtype=torch.uint8).pin_memory()
    h_nb = torch.zeros((N, 2), dtype=torch.int16).pin_memory()
    h_flags = torch.full((N,), 4, dtype=torch.int32).pin_memory()
    h_out = torch.zeros((N, 640), dtype=torch.int16).pin_memory()
    h_ret = torch.zeros((N,), dtype=torch.int32).pin_memory()

    def step_host(t):
        enc.encode_ptr(host_pcm[t].data_ptr(), h_bits.data_ptr(), CAP, h_nb.data_ptr())
        dec.decode_ptr(h_out.data_ptr(), h_bits.data_ptr(), CAP, h_nb.data_ptr(), h_flags.data_ptr(), h_ret.data_ptr())

    for t in range(W):
        step_host(t)
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for t in range(W, T):
        step_host(t)
    torch.cuda.synchronize()
    host_ms = (time.perf_counter() - t0) * 1e3
    if dist:
        t_ = torch.tensor([host_ms], device=dev)
        dist.all_reduce(t_, op=dist.ReduceOp.MAX)
        host_ms = float(t_.item())
    clocks = sampler.stop()
    e2e_value = world * N * K / (host_ms / 1e3)
    checksum = int(h_out.to(torch.int64).sum().item())
    h2d = world * N * (1280 + CAP + 4 + 4)      # whole job, per step: PCM in (encoder) + payload, lengths, flags in (decoder)
    d2h = world * N * (CAP + 4 + 1280 + 4)      # payload + lengths out (encoder) + PCM, return codes out (decoder)

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, torch, N, {
            "device": {"payload": d_bits, "nbytes": d_nb, "pcm": d_out, "ret": d_ret},
            "e2e": {"payload": h_bits, "nbytes": h_nb, "pcm": h_out, "ret": h_ret}})

    if rank == 0:
        peak, peak_src = measured_peaks()
        # per launch: a packet wave is processed as `chunks` launches of each kernel (solo_b200_set_chunks)
        kms = {k: (v[0] / max(v[1], 1)) for k, v in prof.items()}
        kms_wave = {k: v[0] / K for k, v in prof.items()}        # summed launch durations per packet wave (launches overlap)
        n_launch = max(prof["enc_nsq"][1], 1)
        enc_ms = kms["enc_nsq"]
        streams_per_launch = N * K / n_launch
        alg_bytes_enc = streams_per_launch * (1280.0 + mean_payload + 4.0)   # SURVEY.md 8(d): encode reads 1280 B PCM, writes B_out + 4 B
        alg_bytes_dec = N * K / max(prof["decode"][1], 1) * (mean_payload + 4.0 + 4.0 + 1280.0 + 2.0)
        achieved = alg_bytes_enc / (enc_ms / 1e3) / 1e9 if enc_ms > 0 else None
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32",
            "data": "synthetic (speech-replay of the codec's 16 kHz test clip, SURVEY 8(d)(i); fresh codec state)",
            "config": {"workload": "configs[2]: batch=65536 streams/GPU full encode+decode round trip (lostflag 4), 13.6 kb/s",
                       "arithmetic": "int32/int16 fixed point (encoder, SILK decoder), f32 (decoder high band + QMF synthesis)",
                       "streams_per_gpu": N, "streams_total": world * N, "pipeline_chunks": os.environ.get("SOLO_B200_CHUNKS", "default: 1 (device entry points), 3 (host entry points)"), "payload_cap": CAP, "mean_payload_bytes": mean_payload,
                       "l2": "no flush: every step reads a new 84 MB PCM wave and ~0.9 GB of per-stream state (> 126 MB L2)",
                       "parallelism": "streams sharded contiguously across GPUs, no collective on the data path",
                       "host_binding": numa},
            "streams_rt": value / 25.0,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": host_ms / K, "streams_rt": e2e_value / 25.0, "pcm_checksum": checksum},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "sb_enc_nsq_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": (achieved / peak) if achieved else None, "traffic": ncu_traffic("sb_enc_nsq_kernel", streams_per_launch), "peak_source": peak_src,
                         "issue_util": ((ncu_summary() or {}).get("issue_util_time_weighted_pct") or 0) / 100.0 or None,
                         "dram_bytes_per_packet": (ncu_summary() or {}).get("dram_bytes_per_packet"),
                         "warp_inst_per_packet": (ncu_summary() or {}).get("warp_inst_per_packet"),
                         "ncu_capture": (ncu_summary() or {}).get("from"),
                         "algorithmic_bytes_per_launch": alg_bytes_enc, "kernel_ms": enc_ms,
                         "kernel_ms_all": kms, "kernel_ms_per_wave": kms_wave, "streams_per_launch": streams_per_launch,
                         "decode_algorithmic_bytes_per_launch": alg_bytes_dec,
                         "note": "integer-issue / latency bound codec: HBM fraction is small by construction (SURVEY 7.3-1)"},
            "decode_ret_ok": ret_ok,
        }
        if root:
            line["root_ingest"] = root
        if not args.no_cpu_baseline and world == 1:
            cores = usable_cores()
            spt, pk = CPU_SPT, CPU_PK
            res = run_cpu_baseline(cores, spt, pk)
            if res:
                line["cpu_baseline"] = {"value": res["packets_per_s"], "unit": UNIT, "cores": cores, "kind": "reference",
                                        "packets_per_s_per_core": res["packets_per_s"] / cores, "cpus_visible": os.cpu_count(),
                                        "sample": "%d pinned threads (one per usable core) x %d streams x %d packets, same speech-replay input, FIX encode + FLP decode" % (cores, spt, pk)}
            else:
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": cores, "kind": "reference", "sample": "oracle/_ref missing"}
        emit(line)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
