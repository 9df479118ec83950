#!/usr/bin/env python3
"""bench.py — LPCNet synthesis throughput on B200 (driver contract: one JSON line on stdout from rank 0).

  python bench.py --gpus N --steps K --warmup W            # this engine   (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K ...   # the reference's own CPU implementation on the host cores
  python bench.py ... --dump-outputs DIR                    # also write the PCM of the last timed step to DIR/*.npy

Metric (BASELINE.json): synthesized 16 kHz samples/s over batched independent streams.
A "step" = one pass of the hot path over one batch of synthetic feature frames:
  workload `config3_int8`: 4096 streams/GPU x FRAMES frames x 160 samples, int8 block-sparse GRU_A (BASELINE config 3,
  the configuration the metric's ">= 1e8 samples/s/GPU at batch >= 1024 streams" target is quoted on).
`value`  : inputs already resident in HBM, PCM left in HBM, CUDA events on the engine's stream, max over ranks.
`e2e`    : the same step through the host-pointer C-ABI call (lpcnet_b200_batch_synthesize): pinned host features
           -> H2D -> kernels -> D2H PCM, all inside the timed region.
`roofline`: per-sample kernel (the dominant kernel).  Every weight is resident in SHARED MEMORY, so the bound is the
           L1/shared-memory data pipe, not HBM: `bound` = "smem", `achieved` = algorithmic bytes/sample (SURVEY 8d: everything
           run_sample_network must read once per sample) x samples per launch / the kernel's measured duration, `peak` = the
           shared-memory streaming rate MEASURED in this run by the library's micro-kernel (conflict-free LDS.128 on all
           SMs, lpcnet_b200/csrc/microbench.cu).  Because one MMA fetch serves 16 streams the algorithmic figure may exceed the
           physical one; the physical evidence (ncu LSU-pipe %) is quoted beside it.  `sparse_gemv_frac` is the north star's
           own measure (GRU_A weights + indices only).  HBM traffic per sample (ncu) vs the 2.5 B algorithmic is reported too.
`--dump-outputs DIR`: after the timed steps, the PCM the last step of each timed leg returned, as float32 [streams][samples]:
           DIR/pcm.npy (`value` leg, read back from HBM) and DIR/pcm_e2e.npy (`e2e` leg, the host buffer the call filled), with
           DIR/streams.npy, the stream index of every row.  Above DUMP_LIMIT bytes in all, the same seeded sample of streams is
           kept from both.  The inputs and the number of steps before the last one depend only on the arguments, so two builds
           run with the same arguments can be compared array for array.
`cpu_baseline`: the untouched reference compiled by oracle/Makefile (oracle/_ref, timing builds T / TB = -Ofast AVX2/FMA,
           int8 / float) on this box's host cores, one independent stream per usable hardware thread (affinity mask and
           cgroup quota respected), state creation + model load OUTSIDE the timer; plus the 1-core figure.  Falls back to
           the oracle port (kind "port") only if the compiled reference did not travel.
The oracle/reference are used here ONLY as the timed CPU baseline, never as the thing measured for `value`/`e2e`.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import numpy as np

STREAMS_PER_GPU = 4096
FRAMES = 10               # frames per step (1600 samples per stream per step)
LPC_GAMMA = 0.9
METRIC = "16 kHz samples/sec (batched independent streams), whole job"
DUMP_LIMIT = 64 * 10 ** 6  # bytes written by --dump-outputs, all files together
UNIT = "samples/s"


def features_for(n, frames, first_stream=0):
    """DISTINCT synthetic features per stream (SURVEY 8d: seed 1000+s), n streams starting at id `first_stream`."""
    from fixtures import make_feature_batch
    return np.ascontiguousarray(make_feature_batch(range(first_stream, first_stream + n), frames))


def packets_for(n, npackets, first_stream=0):
    """DISTINCT random 8-byte packets per stream (seed 2000+s)."""
    from fixtures import make_packets
    return np.ascontiguousarray(np.stack([make_packets(first_stream + s, npackets) for s in range(n)]))


def host_cpu_info():
    """What the CPU baseline can actually use: affinity mask, cgroup CPU quota, CPU model."""
    try:
        aff = len(os.sched_getaffinity(0))
    except AttributeError:
        aff = os.cpu_count() or 1
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    model = "?"
    try:
        model = [l.split(":")[1].strip() for l in open("/proc/cpuinfo") if l.startswith("model name")][0]
    except Exception:
        pass
    usable = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return {"os_cpu_count": os.cpu_count(), "sched_affinity": aff, "cgroup_cpu_quota": quota, "threads_used": usable, "cpu_model": model}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.lines, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        load = sorted(sm)[len(sm) // 2:]                      # upper half = samples taken under load
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic_per_sample():
    """DRAM bytes per synthesized sample of the per-sample kernel, from the most recent committed `ncu --set full`
    capture (profiles/*_traffic.json, written by tools/ncu_summary.py).  None if no capture is committed."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_traffic.json")))
    if not files:
        return None, None, None
    d = json.load(open(files[-1]))
    return float(d["dram_bytes"]) / float(d["samples_in_launch"]), os.path.basename(files[-1]), d.get("l1_data_pipe_pct_of_peak_active_sms")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_rows(rows, cols, narrays):
    """Stream indices --dump-outputs writes: all of them, or a fixed seeded sample when narrays float32 arrays of
    [rows][cols] and the index list would exceed DUMP_LIMIT."""
    keep = (DUMP_LIMIT - 8 * rows - 4096) // (4 * cols * narrays)        # 4096: the .npy headers
    if keep < 1:
        raise SystemExit("bench: --dump-outputs: one stream's output alone exceeds %d bytes" % DUMP_LIMIT)
    if keep >= rows:
        return np.arange(rows)
    return np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))


def dump_outputs(out_dir, rows, arrays):
    """arrays: name -> int16 PCM [streams][samples]; writes out_dir/<name>.npy (float32, exact for int16) and out_dir/streams.npy."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "streams.npy"), rows.astype(np.float64))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a[rows].astype(np.float32))


# ---------------------------------------------------------------------------------------------------------------------
CPU_WORK = {  # workload -> (reference timing build, blob kind, description)
    "config3_int8": ("T", "int8", "lpcnet_synthesize, int8 AVX2 path (-Ofast -mavx2 -mfma)"),
    "config2_float": ("TB", "float", "lpcnet_synthesize, float path -DDISABLE_DOT_PROD (-Ofast -mavx2 -mfma)"),
    "config5_decode": ("T", "int8", "lpcnet_decode (8-byte packets), int8 AVX2 path (-Ofast -mavx2 -mfma)"),
}


def cpu_reference_run(workload, frames, nthreads):
    """Times the reference's own CPU implementation with one independent stream per thread; state creation and model
    load happen before the clock starts (oracle/ref_shim.c ref_time_streams).  Returns (samples_per_s, kind)."""
    import helpers as H
    build, kind, _ = CPU_WORK[workload]
    decode = workload == "config5_decode"
    blob = H.blob(kind)
    if decode:
        npk = max(1, frames // 4)
        pk = packets_for(nthreads, npk)
        pcm = np.zeros((nthreads, npk * 640), np.int16)
        samples = nthreads * max(0, npk * 4 - 2) * 160
    else:
        feats = features_for(nthreads, frames)
        pcm = np.zeros((nthreads, frames * 160), np.int16)
        samples = nthreads * max(0, frames - 2) * 160       # the first two frames are silent warm-up (no network evaluation)
    if H.have_ref(build):
        L = H.ref_lib(build)
        sec = (L.ref_time_streams(blob, len(blob), None, 0, pk.ctypes.data, npk, nthreads, pcm.ctypes.data) if decode
               else L.ref_time_streams(blob, len(blob), feats.ctypes.data, 20, None, frames, nthreads, pcm.ctypes.data))
        if sec <= 0:
            raise RuntimeError("reference timing run failed")
        return samples / sec, "reference"
    L = H.oracle_lib()
    if decode:
        sec = L.oracle_decode_batch(H.oracle_model(kind), pk.ctypes.data, nthreads, npk, nthreads, pcm.ctypes.data)
    else:
        sec = L.oracle_synthesize_batch(H.oracle_model(kind), feats.ctypes.data, 20, nthreads, frames, nthreads, pcm.ctypes.data)
    return samples / sec, "port"


def cpu_baseline_record(workload, frames=250):
    """All usable host threads + the 1-core figure (BASELINE.md 3) on a bounded sample of the workload."""
    info = host_cpu_info()
    nt = info["threads_used"]
    v1, kind = cpu_reference_run(workload, frames, 1)
    vall, kind = cpu_reference_run(workload, frames, nt)
    return {"value": vall, "unit": UNIT, "cores": nt, "kind": kind, "one_core_value": v1,
            "sample": "%d independent streams (1 per usable host thread) x %d frames, %s; create/load_model outside the timer" % (nt, frames, CPU_WORK[workload][2]),
            "host": info}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    info = host_cpu_info()
    nt = info["threads_used"]
    frames = 250                                            # ~0.15 s of CPU per thread-step at ~2.7e5 samples/s/core
    for _ in range(args.warmup):
        cpu_reference_run(args.workload, 40, nt)
    t0 = time.time()
    vals = []
    for _ in range(args.steps):
        v, kind = cpu_reference_run(args.workload, frames, nt)
        vals.append(v)
    total_s = time.time() - t0
    value = float(np.mean(vals))
    v1, _ = cpu_reference_run(args.workload, frames, 1)
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total_s / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if args.workload == "config2_float" else "u8*s8->s32 (int8 DOT_PROD path) + f32", "data": "synthetic",
        "config": {"workload": "%s on host CPU: one stream per usable host thread, reference src/ compiled by oracle/Makefile; %s" % (args.workload, CPU_WORK[args.workload][2]),
                   "frames_per_step": frames, "streams": nt},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nt, "kind": kind, "one_core_value": v1, "host": info,
                         "sample": "%d independent streams x %d frames per step; create/load_model outside the timer" % (nt, frames)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="config3_int8", choices=["config3_int8", "config2_float", "config5_decode"],
                    help="BASELINE config to run; the default (and the driver's) line is config3_int8")
    ap.add_argument("--streams", type=int, default=0, help="streams per GPU (default: 4096 / 256 / 1024 by workload)")
    ap.add_argument("--frames", type=int, default=FRAMES, help="frames per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the PCM of the last timed step of both legs to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    import helpers as H
    import lpcnet_b200
    if lpcnet_b200.device_count() <= 0:
        raise SystemExit("bench: no CUDA device; this engine has no CPU fallback")
    L = lpcnet_b200.lib()
    n = args.streams or {"config3_int8": STREAMS_PER_GPU, "config2_float": 256, "config5_decode": 1024}[args.workload]
    F = args.frames
    decode = args.workload == "config5_decode"
    if decode:
        F = max(4, F // 4 * 4)                              # whole packets: 4 frames each
    blob = H.blob("float" if args.workload == "config2_float" else "int8")
    batch = lpcnet_b200.Batch(n, blob, lpc_gamma=LPC_GAMMA, device=local, codebooks=H.codebooks() if decode else None)
    algo_total, algo_sparse = batch.algorithmic_bytes()

    if decode:
        feats = packets_for(n, F // 4, first_stream=n * rank)       # "features" = packets [n][F/4][8] uint8, distinct per stream
    else:
        feats = features_for(n, F, first_stream=n * rank)           # distinct per stream (and per rank)
    fbytes, pbytes = feats.nbytes, n * F * 160 * 2
    dump = rank == 0 and args.dump_outputs
    if dump:
        rows = dump_rows(world * n, F * 160, 2)
    L.lpcnet_b200_set_device(local)
    d_feat = L.lpcnet_b200_device_alloc(fbytes)
    d_pcm = L.lpcnet_b200_device_alloc(pbytes)
    assert d_feat and d_pcm
    # N > 1: the one exchange of the path, the PCM gather to rank 0 (SURVEY 8e), is part of EVERY step: rank 0 owns the job's PCM
    # buffer [world*n][F*160]; the other ranks open it through CUDA IPC and set it as their batch's PCM sink, so each finished
    # chunk is pushed there by the rank's copy engine over NVLink inside the call (csrc/batch_api.cu forward_to_sink).  torch
    # only carries the 64-byte handle and the barriers; no framework tensor is on the data path.
    d_gather, gather_opened = None, None
    if dist is not None:
        handle = [None]
        if rank == 0:
            d_gather = L.lpcnet_b200_device_alloc(pbytes * world)
            assert d_gather
            hb = (ctypes.c_ubyte * 64)()
            assert L.lpcnet_b200_ipc_export(d_gather, hb) == 0, L.lpcnet_b200_last_error()
            handle = [bytes(hb)]
        dist.broadcast_object_list(handle, src=0)
        if rank != 0:
            gather_opened = L.lpcnet_b200_ipc_open(handle[0])
            assert gather_opened, L.lpcnet_b200_last_error()
            d_gather = gather_opened
        if os.environ.get("LPCNET_B200_BENCH_DIRECT_SINK"):
            # experiment: the per-sample kernel stores its PCM straight into rank 0's buffer (peer stores over NVLink), no copy at all
            d_pcm_own, d_pcm = d_pcm, d_gather + n * rank * F * 160 * 2
        else:
            batch.set_pcm_sink(d_gather, F * 160, n * rank)
    L.lpcnet_b200_memcpy_h2d(d_feat, feats.ctypes.data, fbytes)
    # pinned host buffers for the e2e leg
    h_feat_p = L.lpcnet_b200_host_alloc(fbytes)
    h_pcm_p = L.lpcnet_b200_host_alloc(pbytes)
    ctypes.memmove(h_feat_p, feats.ctypes.data, fbytes)

    def barrier():
        batch.sync()
        if dist is not None:
            dist.barrier()

    def step_device():
        if decode:
            batch.decode_device(d_feat, F // 4, d_pcm)
        else:
            batch.synthesize_device(d_feat, F, 20, d_pcm)

    def step_e2e():
        r = (L.lpcnet_b200_batch_decode(batch._h, h_feat_p, F // 4, h_pcm_p) if decode
             else L.lpcnet_b200_batch_synthesize(batch._h, h_feat_p, F, 20, 160, h_pcm_p))
        if r != 0:
            raise RuntimeError(L.lpcnet_b200_last_error())

    # the first two frames after a reset are silent and skip the sample loop: consume them before anything is timed
    step_device()
    for _ in range(args.warmup):
        step_device()

    # ---------------- timed: device-resident ----------------
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    wall0 = time.time()
    step_ms, kern_ms, launches = [], [], 0
    for _ in range(args.steps):
        batch.flush_l2()                                     # evict L2 between timed iterations (outside the event bracket)
        batch.timer_start()
        step_device()
        step_ms.append(batch.timer_stop())
        ms, k = batch.last_sample_kernel_ms()
        kern_ms.append(ms); launches += k
    barrier()
    wall = time.time() - wall0
    clk = clocks.stop()
    dev_s = sum(step_ms) * 1e-3
    if dump:                                                 # the last step's PCM: in the job's gather buffer when N > 1
        pcm_dev = np.empty((world * n, F * 160), np.int16)
        L.lpcnet_b200_memcpy_d2h(pcm_dev.ctypes.data, d_gather if dist is not None else d_pcm, pbytes * world)
    # ---------------- timed: end-to-end through the host-pointer C-ABI ----------------
    for _ in range(2):
        step_e2e()
    barrier()
    e2e_ms = []
    for _ in range(args.steps):
        batch.flush_l2(); batch.sync()
        batch.timer_start()                                  # event on the engine's (idle) stream, then H2D -> kernels -> D2H
        step_e2e()                                           # returns after the D2H copy has completed
        e2e_ms.append(batch.timer_stop())
    barrier()
    e2e_s = sum(e2e_ms) * 1e-3
    if dump and dist is None:
        pcm_e2e = np.ctypeslib.as_array(ctypes.cast(h_pcm_p, ctypes.POINTER(ctypes.c_int16)), shape=(n, F * 160)).copy()

    if dist is not None:
        import torch
        t = torch.tensor([dev_s, e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_s, e2e_s = float(t[0]), float(t[1])
        # the gather ran inside every timed step; check what arrived: every rank's shard of the last step must sit in rank 0's
        # buffer bit for bit (digest of the rank's local PCM vs digest of its rows in the gathered buffer)
        import hashlib
        loc = np.ctypeslib.as_array(ctypes.cast(h_pcm_p, ctypes.POINTER(ctypes.c_int16)), shape=(n, F * 160))   # PCM of the last (e2e) step, as returned to the host
        digs = [None] * world
        dist.all_gather_object(digs, hashlib.sha256(loc.tobytes()).hexdigest())
        gather_ok = None
        if rank == 0:
            full = np.empty((world * n, F * 160), np.int16)
            L.lpcnet_b200_memcpy_d2h(full.ctypes.data, d_gather, pbytes * world)
            pcm_e2e = full
            gather_ok = all(hashlib.sha256(full[r * n:(r + 1) * n].tobytes()).hexdigest() == digs[r] for r in range(world))
            if os.environ.get("LPCNET_B200_BENCH_DIRECT_SINK"):
                gather_ok = None                                  # (experiment: the e2e leg does not write the gather buffer)
            else:
                assert gather_ok, "PCM gather: rank 0's buffer does not hold every rank's shard"
        gather_ms = 0.0
    else:
        gather_ms = None

    if dump:
        dump_outputs(args.dump_outputs, rows, {"pcm": pcm_dev, "pcm_e2e": pcm_e2e})
    if rank == 0:
        samples_step = world * n * F * 160
        value = samples_step * args.steps / dev_s
        e2e_value = samples_step * args.steps / e2e_s
        hbm_peak, hbm_src = measured_peaks()
        kms = float(np.mean(kern_ms))                        # per-sample kernel duration per launch (one launch per step here)
        samples_launch = n * F * 160
        achieved = samples_launch * algo_total / (kms * 1e-3) / 1e9
        sparse_achieved = samples_launch * algo_sparse / (kms * 1e-3) / 1e9
        sm_mhz = clk.get("sm_mhz") or 1965.0
        smem_nominal = 128.0 * 148 * sm_mhz * 1e6 / 1e9       # 128 B/clk/SM at the clock observed under load
        smem = lpcnet_b200.measure_smem_peak(local)          # measured in this run (microbench.cu)
        smem_peak = smem["lds128_gbs"]
        tps, tsrc, l1pct = ncu_traffic_per_sample() if args.workload == "config3_int8" else (None, None, None)
        algo_hbm = 2.0 + 20 * 4 / 160.0                        # PCM out + features in per sample (SURVEY 8d)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (fp16-stored weights)" if args.workload == "config2_float" else "u8*s8->s32 (mma.sync IMMA) + f32", "data": "synthetic",
            "config": {"workload": {"config3_int8": "config3_int8: %d streams/GPU x %d frames x 160 samples per step, int8 block-sparse GRU_A, bit-exact vs reference build A",
                                    "config2_float": "config2_float: %d streams/GPU x %d frames x 160 samples per step, float GRU arithmetic with fp16-stored weights, bit-exact vs reference build B",
                                    "config5_decode": "config5_decode: %d streams/GPU x %d frames (8-byte packets -> lpcnet_decode), int8, synthetic VQ codebooks"}[args.workload] % (n, F),
                       "streams_per_gpu": n, "frames_per_step": F, "samples_per_step": samples_step, "parallelism": "streams sharded across GPUs (dp%d), no collective inside the sample loop%s" % (world, "; PCM of every step gathered to rank 0 inside the timed region" if world > 1 else ""),
                       "l2": "256 MiB memset between timed steps (outside the event bracket)", "inputs": "distinct features/packets per stream (seed 1000+s / 2000+s), every stream starts from the reference RNG seed", "x_realtime_per_stream": value / world / n / 16000.0},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(fbytes), "d2h_bytes_per_step": int(pbytes), "ms_per_step": 1e3 * e2e_s / args.steps},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": {"bound": "smem", "achieved": achieved, "peak": smem_peak, "unit": "GB/s", "frac": achieved / smem_peak,
                         "traffic": (tps * samples_launch if tps is not None else None), "traffic_source": tsrc,
                         "peak_source": "measured in this run: conflict-free LDS.128 stream on all SMs (lpcnet_b200_measure_smem_peak, csrc/microbench.cu)",
                         "peak_detail": smem, "smem_peak_gbs_nominal": smem_nominal,
                         "kernel": {"config2_float": "lpcnet_sample_kernel_f32n" if n <= 4 * 148 else "lpcnet_sample_kernel_f32"}.get(args.workload, "lpcnet_sample_kernel"),
                         "kernel_ms_per_launch": kms, "kernel_share_of_step": kms * args.steps / (dev_s * 1e3),
                         "algorithmic_bytes_per_sample": algo_total, "sparse_gemv_bytes_per_sample": algo_sparse,
                         "sparse_gemv_achieved_gbs": sparse_achieved, "sparse_gemv_frac": sparse_achieved / smem_peak,
                         "level_serving_the_bytes": "shared memory (weights resident per SM) + L2 (embedding rows)",
                         "binding_unit": "L1/shared-memory data pipe (LSU wavefronts)", "binding_unit_pct_of_peak_ncu": l1pct,
                         "note": "one MMA operand fetch serves 16 streams, so algorithmic bytes/s can exceed the physical pipe rate; binding_unit_pct_of_peak_ncu is the physical utilisation",
                         "hbm": {"algorithmic_bytes_per_sample": algo_hbm, "dram_bytes_per_sample_ncu": tps,
                                 "achieved_gbs": (tps * samples_launch / (kms * 1e-3) / 1e9 if tps is not None else None),
                                 "peak_gbs": hbm_peak, "peak_source": hbm_src,
                                 "note": "DRAM traffic above the 2.5 B/sample algorithmic figure is the condA/condB/lpc hand-off between the frame-rate kernels and the per-sample kernel; <1 % of the HBM peak either way"}},
            "wall_s_timed_region": wall,
        }
        if gather_ms is not None:
            out["pcm_gather"] = {"in_timed_region": True, "verified": gather_ok, "bytes_per_rank_per_step": int(pbytes), "gathered_bytes_per_step": int(pbytes * world),
                                 "transport": "per-chunk cudaMemcpy2DAsync from each rank's copy engine into rank 0's buffer (CUDA IPC peer mapping, NVLink), "
                                              "enqueued by the C-ABI call itself (lpcnet_b200_batch_set_pcm_sink); value and e2e both include it"}
        if world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_baseline_record(args.workload)
        print(json.dumps(out), flush=True)

    if dist is not None:
        batch.set_pcm_sink(None, 0, 0)
        dist.barrier()                                        # nobody still writes into rank 0's buffer
        if gather_opened:
            L.lpcnet_b200_ipc_close(gather_opened)
        elif d_gather:
            L.lpcnet_b200_device_free(d_gather)
    L.lpcnet_b200_device_free(d_feat)
    L.lpcnet_b200_device_free(d_pcm_own if dist is not None and os.environ.get("LPCNET_B200_BENCH_DIRECT_SINK") else d_pcm)
    L.lpcnet_b200_host_free(h_feat_p); L.lpcnet_b200_host_free(h_pcm_p)
    batch.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
