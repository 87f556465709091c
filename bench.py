#!/usr/bin/env python
"""bench.py - pileup positions/sec through the consensus-inference hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's B200 engine
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path
    python bench.py ... --dump-outputs DIR    # also save a seeded sample of the last timed step's outputs as .npy, so
                                              # that two builds can be compared output for output on identical inputs

Workload (config.workload): BASELINE.json configs[1] - r1041_e82_400bps_sup_v5 consensus on a
synthetic 10 Mb draft: 1111 windows x 10000 pileup columns x 10 features (chunk_len 10000,
overlap 1000; the reference's six 200-window batches coalesced into ONE device batch - the
engine takes any batch size and a B200 holds the whole draft).  One step = one pass of the
hot path over that batch (features in -> probabilities + labels out).  Weights are seeded
synthetic (random-init, the archives in the reference are Git-LFS stubs).

`value`   : positions/s with inputs resident in HBM when the timed region starts
            (mdk_engine_forward_dev), K steps bracketed by CUDA events on the engine stream.
`e2e`     : the same metric through the reference-facing call with HOST buffers
            (mdk_engine_forward: pinned H2D of the features, D2H of probabilities + labels
            inside the timed region).
`roofline`: the dominant kernel, tensor-core bound: algorithmic GRU-gate FLOPs of that kernel per
            launch / its mean launch duration (CUDA events per stage, recorded every step).
N > 1: one process per GPU (torchrun), weights broadcast once over NCCL from rank 0, each rank
runs the same per-GPU workload on its own windows (weak scaling, no data-path collective).
"""
import argparse
import concurrent.futures
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOWS, COLS, FEATS = 1111, 10000, 10
# algorithmic FLOPs per position (SURVEY.md 8d): H=128, F=10, 2 layers, bidirectional
FLOP_REC_PER_LAYER = 2 * (2 * 384 * 128)          # 196 608  (both directions, one layer)
FLOP_INPROJ1 = 2 * (2 * 384 * 256)                # 393 216
FLOP_INPROJ0 = 2 * (2 * 384 * 10)                 # 15 360
FLOP_GRU_TOTAL = 2 * FLOP_REC_PER_LAYER + FLOP_INPROJ1 + FLOP_INPROJ0   # 801 792


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return {"hbm_gbs": d["hbm_gbs"], "tflops_burst": d["bf16_tflops"],
                "tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "tflops_burst": 1590.0, "tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None
        self.nvml = None
        self.samples = []          # (sm MHz, reason bits, power W) from the NVML poller
        self.stop_flag = False

    def start(self):
        # NVML poller (a sample every ~10 ms: the timed region of a default run lasts a few hundred ms); nvidia-smi -lms
        # is the fallback when the binding is missing
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.device
            if vis:
                try:
                    idx = int(vis.split(",")[self.device])
                except (ValueError, IndexError):
                    idx = self.device
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml = pynvml
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _poll(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)
                bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
                except Exception:
                    watts = None
                self.samples.append((float(mhz), int(bits), watts))
            except Exception:
                break
            time.sleep(0.01)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            nv = self.nvml
            self.stop_flag = True
            self.thread.join(timeout=2)
            try:
                smax = float(nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM))
            except Exception:
                smax = None
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                     "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                     "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            sm = [x[0] for x in self.samples]
            reasons = sorted(k for k, bit in names.items() if any(x[1] & bit for x in self.samples))
            watts = [x[2] for x in self.samples if x[2] is not None]
            out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "samples": len(sm),
                   "reasons": reasons, "source": "nvml"}
            if sm:
                out["sm_mhz_min"] = min(sm)
            if watts:
                out["power_w"] = statistics.median(watts)
            return out
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def host_cores():
    """Host threads this process may really use: scheduler affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


# stdout carries exactly ONE line (the JSON): libraries that chat on fd 1 (NCCL prints its version there under torchrun)
# are sent to stderr for the whole run, and the line is written to the saved descriptor at the end
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def log(msg):
    print("[bench %.1fs] %s" % (time.perf_counter() - T_START, msg), file=sys.stderr, flush=True)


T_START = time.perf_counter()


def fill_features(x, seed):
    """Fill a float32 [B,T,F] array IN PLACE with normalised-count-like values (rows sum to 1)."""
    rng = np.random.default_rng(seed)
    rng.random(out=x.reshape(-1), dtype=np.float32)
    step = max(1, (1 << 22) // (x.shape[1] * x.shape[2]))
    for i in range(0, x.shape[0], step):
        b = x[i:i + step]
        b *= b * b
        b /= b.sum(axis=-1, keepdims=True)
    return x


def cpu_reference_rate(threads, sample_windows, cols, feats, steps=1, warmup=0, budget_s=12.0):
    """positions/s of the reference's CPU arithmetic (torch fp32 nn.GRU + Linear + softmax, the
    oracle restatement of medaka/architectures/gru.py + models.py:303-313) on a bounded sample.

    ``cols`` <= 0 picks the number of columns so that one pass takes about ``budget_s`` seconds
    (calibrated on a 20-column probe); per-position cost does not depend on the window length.
    Returns (positions/s, seconds per step, cols used)."""
    import torch
    from oracle import gru_oracle, synth
    torch.set_num_threads(threads)
    sd = synth.synth_state_dict(0, num_features=feats)
    model = gru_oracle.build(sd, num_features=feats)
    if cols <= 0:
        probe = fill_features(np.empty((sample_windows, 20, feats), dtype=np.float32), 2)
        gru_oracle.predict_on_batch(model, probe)
        t0 = time.perf_counter()
        gru_oracle.predict_on_batch(model, probe)
        r0 = sample_windows * 20 / (time.perf_counter() - t0)
        cols = int(min(2000, max(40, r0 * budget_s / sample_windows)))
    x = fill_features(np.empty((sample_windows, cols, feats), dtype=np.float32), 1)
    for _ in range(warmup):
        gru_oracle.predict_on_batch(model, x[:, :min(cols, 500)])      # thread pool / allocator warm-up on a short slice
    t0 = time.perf_counter()
    for _ in range(steps):
        gru_oracle.predict_on_batch(model, x)
    dt = time.perf_counter() - t0
    return steps * sample_windows * cols / dt, dt / steps, cols


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path on this box's host cores (rank 0 only)."""
    if rank != 0:
        return
    cores = host_cores()
    sample_windows = args.cpu_windows
    rate, sec_per_step, cols = cpu_reference_rate(cores, sample_windows, args.cpu_cols, FEATS, steps=args.steps,
                                                  warmup=min(args.warmup, 1))
    sample = "%d windows x %d cols per step (the reference's 200-window batch, truncated in time)" % (
        sample_windows, cols)
    line = {
        "impl": "reference", "metric": "pileup positions/sec (consensus inference)", "value": rate,
        "unit": "positions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config), "baseline_config": args.config,
                   "timing": "host wall clock, CPU only", "threads": cores},
        "cpu_baseline": {"value": rate, "unit": "positions/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": rate, "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


CONFIGS = {
    # BASELINE.json configs[1..4]: windows per GPU, columns per window, features, what a step is
    2: dict(windows=1111, cols=10000, feats=10,
            name="r1041_e82_400bps_sup_v5 consensus, synthetic 10 Mb draft: 1111 windows x 10000 cols x 10 feats "
                 "(chunk_len 10000, overlap 1000)"),
    3: dict(windows=2778, cols=10000, feats=10,
            name="r1041_e82_400bps_sup_v5 consensus, synthetic 200 Mb draft region-sharded over 8 GPUs: this rank's share, "
                 "2778 of 22223 windows x 10000 cols x 10 feats"),
    4: dict(windows=5556, cols=10000, feats=10,
            name="r1041_e82_400bps_sup_variant_v5, synthetic 50 Mb: 5556 windows x 10000 cols x 10 feats; the variant decode "
                 "of a step's output (mdk_decode_variants) is timed additionally, see variant_decode"),
    5: dict(windows=1111, cols=10000, feats=20,
            name="r941_min_hac_g507-style legacy encoder, synthetic 10 Mb: 1111 windows x 10000 cols x 20 feats (two "
                 "datatypes, normalise='fwd_rev'); a step starts from raw uint64 counts (normalise kernel + forward)"),
}


def variant_leg(probs, B, T, dev):
    """BASELINE config 4's extra: the variant decode of one step's probabilities (argmax with gaps, variant-column rule,
    run detection, quality sums: medaka/labels.py:889-1014) on the GPU through host buffers, per 512-window joined
    sample, beside the numpy restatement on a bounded sample."""
    from medaka_b200 import labels as mlabels
    from oracle import variants_oracle
    rs = np.random.RandomState(5)
    vminor = (rs.uniform(size=T) < 0.12).astype(np.int64)       # synthetic draft: ~12 % insertion columns
    vminor[0] = 0
    vref = np.where(vminor == 0, rs.randint(1, 5, T), 0).astype(np.uint8)

    def gpu_pass():
        n_var = 0
        for w in range(0, B, 512):
            wb = min(B, w + 512)
            mn, rf = np.tile(vminor, wb - w), np.tile(vref, wb - w)
            n_var += len(mlabels.decode_variant_arrays(probs[w:wb].reshape(-1, 5), mn, rf, dev, want_quals=False)["run_start"])
        return n_var
    gpu_pass()
    t0 = time.perf_counter()
    n_var = gpu_pass()
    t_gpu = time.perf_counter() - t0
    # numpy restatement (oracle/variants_oracle.py) on 8 windows
    nw = min(B, 8)
    major = np.cumsum(vminor == 0) - 1
    pos = np.empty(T, dtype=[("major", "<i8"), ("minor", "<i8")])
    pos["major"], pos["minor"] = major, vminor
    draft = "".join("*ACGT"[c] for c in vref[vminor == 0])
    t0 = time.perf_counter()
    for w in range(nw):
        variants_oracle.decode_variants(pos, probs[w], draft)
    t_cpu = time.perf_counter() - t0
    return {"columns_per_step": int(B) * int(T), "gpu_ms_per_step": t_gpu * 1e3, "gpu_columns_per_s": B * T / t_gpu,
            "variant_runs": int(n_var), "cpu_columns_per_s": nw * T / t_cpu,
            "cpu_sample": "%d windows, numpy restatement incl. Variant record building" % nw,
            "note": "timed separately from the inference legs (medaka vcf is a separate consumer of the stored probabilities)"}


def workload_name(cfg=2):
    return CONFIGS[cfg]["name"]


DUMP_BYTES = 48 << 20      # --dump-outputs: probabilities + labels, both as float32 (24 bytes per position)


def dump_selection(B, T):
    """Windows (a fixed seeded sample, sorted) and leading columns per window whose outputs fit in DUMP_BYTES."""
    cols = min(T, DUMP_BYTES // 24)
    n = max(1, min(B, DUMP_BYTES // (24 * cols)))
    return np.sort(np.random.default_rng(0).choice(B, n, replace=False)), cols


def copy_outputs(lm, dev, d_probs, d_labels, T, windows, cols):
    """The sampled part of one step's device outputs ([B,T,5] float32 probabilities, [B,T] uint8 labels) on the host."""
    lib, ffi = lm.lib, lm.ffi
    probs = np.empty((len(windows), cols, 5), dtype=np.float32)
    labels = np.empty((len(windows), cols), dtype=np.uint8)
    for i, w in enumerate(windows):
        lm.check(lib.mdk_memcpy_d2h(dev, ffi.from_buffer(probs[i]), ffi.cast("float *", d_probs) + int(w) * T * 5,
                                    probs[i].nbytes))
        lm.check(lib.mdk_memcpy_d2h(dev, ffi.from_buffer(labels[i]), ffi.cast("uint8_t *", d_labels) + int(w) * T,
                                    labels[i].nbytes))
    return probs, labels


def write_outputs(out_dir, probs, labels, windows):
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "probs.npy"), probs)
    np.save(os.path.join(out_dir, "labels.npy"), labels.astype(np.float32))
    np.save(os.path.join(out_dir, "windows.npy"), windows.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json config (2..5)")
    ap.add_argument("--windows", type=int, default=0, help="windows per step per GPU (0 = the config's)")
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--batch-windows", type=int, default=200,
                    help="windows per predict_on_batch call in the e2e leg (the reference's --batch_size; the engine "
                         "coalesces them into device-filling groups)")
    ap.add_argument("--rec-mode", default="auto", choices=["auto", "one", "pp"])
    ap.add_argument("--precision", default="tc", choices=["tc", "fp32"])
    ap.add_argument("--cpu-windows", type=int, default=200, help="windows in the bounded CPU-baseline sample")
    ap.add_argument("--cpu-cols", type=int, default=0,
                    help="columns per window in the CPU sample (0 = the full window length for the cpu_baseline of the "
                         "default run, ~15 s; sized for ~12 s per step for --impl reference)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's probabilities and labels (rank 0, a seeded sample of at most "
                         "48 MB) and the sampled window indices as DIR/{probs,labels,windows}.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")

    capture_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = CONFIGS[args.config]
    global FEATS
    FEATS = cfg["feats"]

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    from medaka_b200 import libmedaka as lm
    from medaka_b200 import models
    from oracle import synth   # seeded synthetic weights/inputs + the cpu_baseline leg only

    lib = lm.load()
    ffi = lm.ffi
    dev = local_rank if world > 1 else 0
    info = lm.require_gpu(dev)
    sm_count = int(info["sm_count"])

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(dev)
        dist.init_process_group("nccl", device_id=torch.device("cuda", dev))

    # ---- weights: rank 0 owns them, one NCCL broadcast of the packed fp32 blob (1.62 MB) ----
    F = cfg["feats"]
    sd = synth.synth_state_dict(0, num_features=F)
    keys = sorted(sd)
    if world > 1:
        blob = np.concatenate([sd[k].ravel() for k in keys])
        t = torch.from_numpy(blob if rank == 0 else np.zeros_like(blob)).cuda()
        dist.broadcast(t, src=0)
        flat = t.cpu().numpy()
        off = 0
        for k in keys:
            n = sd[k].size
            sd[k] = flat[off:off + n].reshape(sd[k].shape).copy()
            off += n
    model = models.GRUModel(num_features=F, device=dev)
    model.load_state_dict(sd)
    model.set_precision(args.precision)
    model.set_rec_mode(args.rec_mode)
    eng = model.engine

    B = args.windows or cfg["windows"]
    T = args.cols or cfg["cols"]
    P = B * T
    group = model.preferred_batch_size()                 # windows per device forward (one wave; lanes alternate)
    chunks = [(a, min(B, a + group)) for a in range(0, B, group)]
    log("config %d: %d x %d x %d synthetic features into pinned host memory" % (args.config, B, T, F))
    feats = fill_features(model.pinned("bench_feats", (B, T, F), np.float32), 1000 + rank)
    log("reserving the compute lanes (%d-window groups)" % min(group, B))
    model.reserve(min(group, B), T)

    def dalloc(nbytes):
        pp = ffi.new("void **")
        lm.check(lib.mdk_dev_alloc(dev, nbytes, pp))
        return pp[0]

    # ---- device-resident leg ("value"): inputs in HBM when the timed region starts ----
    d_feats = dalloc(feats.nbytes)
    lm.check(lib.mdk_memcpy_h2d(dev, d_feats, ffi.from_buffer(feats), feats.nbytes))
    # two output sets: consecutive steps run on alternating lanes and may overlap
    d_probs_set = [dalloc(P * 5 * 4), dalloc(P * 5 * 4)]
    d_labels_set = [dalloc(P), dalloc(P)]
    d_probs, d_labels = d_probs_set[0], d_labels_set[0]
    d_counts = d_major = d_minor = d_depth = None
    if args.config == 5:
        # raw counts resident in HBM: the step is normalise (a3) + forward; counts chosen so that the features are the
        # synthetic ones is not possible bit-for-bit, so the normalise output simply replaces d_feats
        counts, pos = synth.synth_counts(min(P, 4000000), seed=77, num_dtypes=2)
        reps = (P + len(counts) - 1) // len(counts)
        counts = np.tile(counts, (reps, 1))[:P]
        major = np.tile(pos["major"], reps)[:P].astype(np.int64)
        minor = np.tile(pos["minor"], reps)[:P].astype(np.int64)
        minor[0] = 0
        d_counts, d_major, d_minor, d_depth = dalloc(counts.nbytes), dalloc(P * 8), dalloc(P * 8), dalloc(P * 8)
        lm.check(lib.mdk_memcpy_h2d(dev, d_counts, ffi.from_buffer(counts), counts.nbytes))
        lm.check(lib.mdk_memcpy_h2d(dev, d_major, ffi.from_buffer(major), P * 8))
        lm.check(lib.mdk_memcpy_h2d(dev, d_minor, ffi.from_buffer(minor), P * 8))
        del counts

    step_no = [0]

    def step_dev():
        d_probs, d_labels = d_probs_set[step_no[0] & 1], d_labels_set[step_no[0] & 1]
        step_no[0] += 1
        if args.config == 5:
            lm.check(lib.mdk_device_synchronize(dev))    # the normalise kernel runs on the default stream
            lm.check(lib.mdk_normalise_counts_dev(dev, ffi.cast("const uint64_t *", d_counts),
                                                  ffi.cast("const int64_t *", d_major), ffi.cast("const int64_t *", d_minor),
                                                  P, 2, lib.MDK_NORM_FWD_REV, 0, ffi.cast("float *", d_feats),
                                                  ffi.cast("int64_t *", d_depth)))
            lm.check(lib.mdk_device_synchronize(dev))
        for a, b in chunks:
            lm.check(lib.mdk_engine_forward_dev(
                eng, ffi.cast("const float *", d_feats) + a * T * F, b - a, T, ffi.cast("float *", d_probs) + a * T * 5,
                ffi.NULL, ffi.cast("uint8_t *", d_labels) + a * T))

    def barrier():
        if dist is not None:
            dist.barrier()
        lm.check(lib.mdk_engine_sync(eng))

    log("device-resident leg: warm-up")
    for _ in range(args.warmup):
        step_dev()
    barrier()
    log("device-resident leg: timing %d steps" % args.steps)
    launches0 = model.launch_count()
    sampler = ClockSampler(dev)
    sampler.start()
    ms = ffi.new("float *")
    lm.check(lib.mdk_engine_timer_start(eng))
    for _ in range(args.steps):
        step_dev()
    lm.check(lib.mdk_engine_timer_stop(eng, ms))     # end event after every lane and the copy streams
    barrier()
    clocks = sampler.stop()
    dumped = None
    if args.dump_outputs and rank == 0:
        # copied now: the forwards below write into the same output sets
        last = (step_no[0] - 1) & 1
        dump_windows, dump_cols = dump_selection(B, T)
        dumped = copy_outputs(lm, dev, d_probs_set[last], d_labels_set[last], T, dump_windows, dump_cols)
    dev_ms = float(ms[0])
    launches = model.launch_count() - launches0 + (args.steps if args.config == 5 else 0)
    tm = ffi.new("mdk_timings *")
    n_fwd = min(args.steps * len(chunks), 32)
    lm.check(lib.mdk_engine_mean_timings(eng, n_fwd, tm))
    stage = {k: float(getattr(tm, k)) for k in ("inproj0_ms", "rec0_ms", "inproj1_ms", "rec1_ms", "head_ms")}

    # sanity: the timed path produced real outputs (labels consistent with probabilities)
    chk = np.empty((min(B, 4), T, 5), dtype=np.float32)
    lm.check(lib.mdk_memcpy_d2h(dev, ffi.from_buffer(chk), d_probs, chk.nbytes))
    assert np.isfinite(chk).all() and abs(float(chk.sum(-1).mean()) - 1.0) < 1e-4

    # one forward on an otherwise idle GPU: clean per-kernel durations (in the timed region the groups of two lanes
    # overlap, so a kernel's event-to-event time there includes the other lane's kernels)
    b0 = chunks[0][1]
    barrier()
    lm.check(lib.mdk_engine_forward_dev(eng, ffi.cast("const float *", d_feats), b0, T, ffi.cast("float *", d_probs),
                                        ffi.NULL, ffi.cast("uint8_t *", d_labels)))
    lm.check(lib.mdk_engine_mean_timings(eng, 1, tm))
    solo = {k: float(getattr(tm, k)) for k in ("inproj0_ms", "rec0_ms", "inproj1_ms", "rec1_ms", "head_ms")}

    # the recurrent kernel with one CTA on every SM, alone on the GPU: a full wave of windows (2368 for the two-tile
    # kernel) over as many columns as the reserved workspace holds - the per-step cost of the persistent kernel does
    # not depend on the window length
    full_wave = None
    if args.precision == "tc" and args.config != 5:
        tiles_b0 = (b0 + 15) // 16
        pp_sel = args.rec_mode == "pp" or (args.rec_mode == "auto" and tiles_b0 * 2 > sm_count // 2)
        fw_windows = 16 * sm_count if pp_sel else 8 * sm_count
        fw_cols = (b0 * T) // fw_windows
        if fw_cols >= 256:
            model.set_rec_mode("pp" if pp_sel else "one")
            for _ in range(2):
                lm.check(lib.mdk_engine_forward_dev(eng, ffi.cast("const float *", d_feats), fw_windows, fw_cols,
                                                    ffi.cast("float *", d_probs), ffi.NULL, ffi.cast("uint8_t *", d_labels)))
                barrier()
            lm.check(lib.mdk_engine_mean_timings(eng, 1, tm))
            model.set_rec_mode(args.rec_mode)
            fw_ms = 0.5 * (float(tm.rec0_ms) + float(tm.rec1_ms))
            fw_tf = fw_windows * fw_cols * FLOP_REC_PER_LAYER / (fw_ms * 1e-3) / 1e12
            pk = measured_peaks()
            full_wave = {"windows": fw_windows, "cols": fw_cols, "ctas": sm_count, "rec0_ms": float(tm.rec0_ms),
                         "rec1_ms": float(tm.rec1_ms), "inproj1_ms": float(tm.inproj1_ms), "achieved": fw_tf,
                         "peak": pk["tflops_burst"], "frac": fw_tf / pk["tflops_burst"],
                         "peak_source": "MEASURED_PEAKS.json bf16 burst (kernel timed alone)"}

    # ---- host-buffer leg ("e2e"): the reference-facing call with HOST buffers, the way run_prediction drives it -
    # batches of --batch-windows windows (the reference's --batch_size) submitted with a look-ahead
    # (mdk_engine_submit / mdk_engine_wait); every step copies its features in and its probabilities + labels out ----
    bw = max(1, min(args.batch_windows, B))
    batches = [(a, min(B, a + bw)) for a in range(0, B, bw)]
    depth = model.lookahead(bw, T)
    n_slots = 2
    h_probs = model.pinned("bench_probs", (n_slots, B, T, 5), np.float32)   # results stay valid while the next step is
    h_labels = model.pinned("bench_labels", (n_slots, B, T), np.uint8)      # already queued

    def run_host(n):
        # the reference-facing loop (medaka/prediction.py:44-52): batches submitted with the engine's look-ahead, results
        # collected in order
        pending = []
        for k in range(n):
            for a, b in batches:
                while len(pending) >= depth:
                    model.wait(pending.pop(0))
                pending.append(model.submit_arrays(feats[a:b], h_probs[k % n_slots, a:b], h_labels[k % n_slots, a:b]))
        while pending:
            model.wait(pending.pop(0))

    log("host-buffer leg (%d-window batches, %d in flight)" % (bw, depth))
    run_host(max(1, min(args.warmup, 2)))
    barrier()
    lm.check(lib.mdk_engine_timer_start(eng))
    run_host(args.steps)
    lm.check(lib.mdk_engine_timer_stop(eng, ms))
    barrier()
    e2e_ms = float(ms[0])
    assert np.isfinite(h_probs[(args.steps - 1) % n_slots, :2]).all()

    if dist is not None:
        t = torch.tensor([dev_ms, e2e_ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)     # max over ranks, device-timed
        dev_ms, e2e_ms = float(t[0]), float(t[1])

    total_positions = world * args.steps * P
    value = total_positions / (dev_ms * 1e-3)
    e2e = total_positions / (e2e_ms * 1e-3)

    # ---- roofline of the dominant kernel (tensor bound) ----
    # The recurrent kernel of a config-2 group runs on a PART of the GPU (ping-pong kernel: one CTA per window tile =
    # 70 of 148 SMs for 1111 windows; the other lane's kernels use the rest), so its roofline is the tensor peak of the
    # SMs it holds: peak = sustained bf16 peak x CTAs / SMs.  achieved = algorithmic FLOPs per launch / mean launch
    # duration in the TIMED REGION (event to event on the launching stream; includes any wait for SMs, so it is a lower
    # bound).  full_wave_solo is the same kernel launched alone with one CTA on every SM.
    peaks = measured_peaks()
    p0 = b0 * T
    tiles0 = (b0 + 15) // 16
    use_pp = args.precision == "tc" and (args.rec_mode == "pp" or (args.rec_mode == "auto" and tiles0 * 2 > sm_count // 2))
    rec_ctas = tiles0 if use_pp else min(2 * tiles0, sm_count)
    sm_share = min(1.0, rec_ctas / float(sm_count))
    rec_ms_region = 0.5 * (stage["rec0_ms"] + stage["rec1_ms"])
    kernels = {
        "recurrent kernel (%s: GRU recurrence, layer-0 and layer-1 launches)" % ("rec_pp_kernel" if use_pp else "rec_tc_kernel"):
            (rec_ms_region, p0 * FLOP_REC_PER_LAYER, solo["rec0_ms"] + solo["rec1_ms"], sm_share),
        "gemm_tc_kernel (layer-1 input projection)": (stage["inproj1_ms"], p0 * FLOP_INPROJ1, solo["inproj1_ms"], 1.0),
    }
    dom = max(kernels, key=lambda k: kernels[k][2])
    k_ms, k_flop, k_share_ms, k_sms = kernels[dom]
    achieved = k_flop / (k_ms * 1e-3) / 1e12
    peak = peaks["tflops_sustained"] * k_sms
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if args.config == 2 and args.precision == "tc" and os.path.exists(tpath):
        with open(tpath) as fh:
            tj = json.load(fh)
        traffic = tj.get(("rec_pp_kernel" if use_pp else "rec_tc_kernel") if dom.startswith("recurrent") else "gemm_tc_kernel")
    flop_gru = 2 * FLOP_REC_PER_LAYER + FLOP_INPROJ1 + 2 * (2 * 384 * F)
    roofline = {
        "bound": "tensor", "kernel": dom, "achieved": achieved, "peak": peak,
        "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
        "peak_source": ("MEASURED_PEAKS.json bf16 sustained (kernel timed inside a long step) x %d/%d SMs the launch occupies"
                        % (round(k_sms * sm_count), sm_count)) if peaks["source"] == "measured" else "fallback (B200_PROFILING.md)",
        "launch": {"windows": b0, "cols": T, "ctas": rec_ctas if dom.startswith("recurrent") else None,
                   "flop_per_launch": k_flop, "mean_ms_in_timed_region": k_ms},
        "note": "algorithmic FLOPs; operands are fp16 hi/lo pairs so the kernel issues 3 MMAs per product "
                "(fp32-faithful parity), i.e. executed tensor FLOPs are 3x this figure",
        "kernel_share_of_step": k_share_ms / max(sum(solo.values()), 1e-9),
        "solo_stage_ms": solo, "solo_windows": b0,
        "timed_region_stage_ms": stage,
        "full_wave_solo": full_wave,
        "whole_pipeline_achieved": value / world * flop_gru / 1e12,
        "whole_pipeline_frac": value / world * flop_gru / 1e12 / peaks["tflops_sustained"],
        "whole_pipeline_note": "all GRU-gate FLOPs (both recurrences + the layer-1 projection, all three on the tensor "
                               "cores) / step time of the timed region, against the sustained bf16 peak",
    }

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    cpu_baseline = None
    if not args.no_cpu_baseline:
        cores = host_cores()
        log("cpu baseline on %d threads" % cores)
        rate, sec, ccols = cpu_reference_rate(cores, args.cpu_windows, args.cpu_cols or T, F, steps=1, warmup=1)
        cpu_baseline = {"value": rate, "unit": "positions/s", "cores": cores, "kind": "port",
                        "sample": "%d windows x %d cols, 1 warm-up + 1 timed pass (%.1f s), torch %s fp32 nn.GRU oracle" % (
                            args.cpu_windows, ccols, sec, torch.__version__)}
    log("done")

    line = {
        "metric": "pileup positions/sec (consensus inference)", "value": value, "unit": "positions/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(args.config) if not (args.windows or args.cols) else
                   "synthetic %d windows x %d cols x %d feats" % (B, T, F),
                   "baseline_config": args.config, "windows_per_gpu": B, "cols": T, "features": F,
                   "precision": args.precision, "rec_mode": args.rec_mode,
                   "arithmetic": "fp32 state, gate math and accumulation; tensor-core operands as fp16 hi/lo pairs, three "
                                 "products per contraction (fp32-faithful)" if args.precision == "tc" else "fp32 CUDA cores",
                   "group_windows": min(group, B), "batch_windows": bw, "batches_in_flight": depth,
                   "l2_policy": "inputs larger than L2 (%d MB of features, > 3 GB of activations per step)" % (feats.nbytes >> 20),
                   "sm_count": info["sm_count"]},
        "e2e": {"value": e2e, "unit": "positions/s", "h2d_bytes_per_step": int(feats.nbytes),
                "d2h_bytes_per_step": int(P * 5 * 4 + P), "ms_per_step": e2e_ms / args.steps,
                "batch_windows": bw},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "cpu_baseline": cpu_baseline,
    }
    if args.config == 4:
        line["variant_decode"] = variant_leg(h_probs[(args.steps - 1) % n_slots], B, T, dev)
    if dumped is not None:
        write_outputs(args.dump_outputs, *dumped, dump_windows)
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
