#!/usr/bin/env python3
"""bench.py -- MFCC frames/s (48 kHz, n_fft=2048, hop=512, 128 mel, 40 coefficients) on N B200s.

Usage (DESIGN.md section 6):
  python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun, one rank per GPU)
  python bench.py --impl reference ...                     (the reference's own CPU path, oracle/_ref)
  python bench.py ... --dump-outputs DIR                   (also write the MFCCs of the last timed step to DIR/mfcc.npy)
One JSON line on stdout from rank 0.  K is the number of timed steps of every timed loop.

A "step" is one pass of the fused STFT->mel->log->DCT path over one synthetic batch:
  N=1 : BASELINE config 2 = 1024 clips x 5 s (983 MB of samples, larger than the 126 MB L2).
  N>1 : the same 1024 clips PER GPU (weak scaling, config 5 at N=8) with the all-gather of the (1024, 465, 40)
        result blocks -- the path's only exchange step -- fused into the kernel epilogue as NVLink P2P stores
        (--gather peer, default) or done by NCCL on a side stream (--gather nccl).
`value` is device-timed (CUDA events on the launching stream) with inputs resident in HBM;
`e2e` goes through the public call with pinned HOST buffers, H2D and D2H inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.realpath(__file__))
_REAL_STDOUT = None


def emit(obj):
    """The one JSON line of the contract, on the process's original stdout."""
    text = json.dumps(obj) + "\n"
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, text.encode())

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SR, RADIX, NFFT, HOP, NMEL, NCC = 48000, 11, 2048, 512, 128, 40
CLIP_SECONDS = 5
L = SR * CLIP_SECONDS
T = (L - NFFT) // HOP + 1
BATCH_PER_GPU = 1024
# algorithmic (compulsory) HBM bytes per clip: every sample read once + result written once (SURVEY 8d)
BYTES_PER_CLIP = 4 * L + 4 * T * NCC
BYTES_PER_FRAME_READ_MODEL = 4 * NFFT + 4 * NCC     # north-star "each frame reads its window" accounting
FLOP_PER_FRAME = 75e3
# BASELINE configs 3 and 4 (reported as extra keys of the same JSON line at N = 1)
CQT_BATCH, CQT_NUM = 1024, 84
CWT_BATCH, CWT_NUM, CWT_RADIX, CWT_SAMPLES = 512, 84, 19, SR * 10      # 10 s = 480 000 samples, zero-padded to 2^19


def ncu_traffic(summary_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, parsed from a committed ncu summary under profiles/
    (Mbyte / Gbyte units as ncu prints them); None when the file or the two metrics are missing."""
    path = os.path.join(ROOT, "profiles", summary_name)
    try:
        tot, seen = 0.0, 0
        for line in open(path):
            f = line.split()
            if len(f) >= 3 and f[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[f[2]]
                tot += float(f[1]) * unit
                seen += 1
        return int(tot) if seen == 2 else None
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}, "fallback"


class ClockSampler:
    """SM clock and throttle reasons polled every ~5 ms through NVML (nvidia-smi every 200 ms as a fallback) in a side
    thread; `mark()` brackets the timed region and the reported median / reasons come from the samples inside it."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index=0):
        self.index, self.rows, self.proc, self.nvml = index, [], None, None
        self.t0 = self.t1 = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def mark(self, begin):
        """brackets the timed region; one synchronous NVML sample is taken just inside each end so that even a region of a
        few milliseconds (shorter than the polling thread's wake-up) carries clock / throttle evidence"""
        if begin:
            self.t0 = time.perf_counter()
            self._sample_now()
        else:
            self._sample_now()
            self.t1 = time.perf_counter()

    def _sample_now(self):
        n = self.nvml
        if n is None:
            return
        try:
            mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.rows.append((time.perf_counter(), mhz, self.max_mhz, mask))
        except Exception:
            pass

    def _poll(self):
        n = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
                try:
                    mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                except Exception:
                    mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
                self.rows.append((time.perf_counter(), mhz, self.max_mhz, mask))
            except Exception:
                pass
            time.sleep(0.004)

    def _read(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                mask = sum(bit for (name, bit), v in zip((("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40),
                                                           ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)), r[5:9])
                           if v.lower().startswith("active"))
                self.rows.append((time.perf_counter(), float(r[1]), float(r[2]), mask))
            except Exception:
                continue

    def stop(self):
        if self.nvml is None and not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=1)
        else:
            time.sleep(0.25)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        inside = [r for r in self.rows if self.t0 is not None and self.t1 is not None and self.t0 <= r[0] <= self.t1]
        use = inside if inside else self.rows
        reasons = sorted(name for name, bit in self.BITS.items() if any(r[3] & bit for r in use))
        return {"sm_mhz": float(np.median([r[1] for r in use])) if use else None,
                "sm_max_mhz": max(r[2] for r in use) if use else None,
                "samples": len(use), "samples_in_timed_region": len(inside), "samples_total": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi", "reasons": reasons}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each (clips, ...) result as out_dir/<name>.npy in float32.  A result larger than its share of DUMP_BYTES is
    cut to a fixed sample of clips (numpy seed 0, ascending clip order), the same for every run with the same --batch /
    --gpus, so that two builds can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays)
    for name, a in arrays.items():
        n = a.shape[0]
        per_clip = 4 * a[0].numel()
        if n * per_clip > budget:
            keep = np.sort(np.random.default_rng(0).choice(n, budget // per_clip, replace=False))
            a = a[keep]
        np.save(os.path.join(out_dir, name + ".npy"), a.float().cpu().numpy())


# --------------------------------------------------------------------------- reference / CPU arm
def _cpu_worker(args):
    lib_path, seed, clips, warm = args
    import ctypes
    sys.path.insert(0, ROOT)
    import audioflux_b200 as af
    from audioflux_b200 import capi
    lib = ctypes.CDLL(lib_path)
    capi.bind(lib)
    S, D = af.SpectralFilterBankScaleType, af.SpectralDataType
    b = af.BFT(NMEL, RADIX, SR, slide_length=HOP, scale_type=S.MEL, data_type=D.POWER, _lib=lib)
    xx = af.XXCC(NMEL, _lib=lib)
    x = (0.1 * np.random.default_rng(seed).standard_normal((clips, L))).astype(np.float32)
    for i in range(warm):
        mel, _ = b.bft_planes(x[i % clips], 1)
        xx.xxcc_planes(mel, NCC)
    t0 = time.perf_counter()
    for i in range(clips):
        mel, _ = b.bft_planes(x[i], 1)
        xx.xxcc_planes(mel, NCC)
    return time.perf_counter() - t0


def cpu_info():
    """CPU model, logical cores of this process's affinity mask and physical cores (from /proc/cpuinfo)."""
    model, phys = "unknown", set()
    try:
        pid = cid = None
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name") and model == "unknown":
                model = line.split(":", 1)[1].strip()
            elif line.startswith("physical id"):
                pid = line.split(":", 1)[1].strip()
            elif line.startswith("core id"):
                cid = line.split(":", 1)[1].strip()
                phys.add((pid, cid))
    except Exception:
        pass
    try:
        logical = len(os.sched_getaffinity(0))
    except Exception:
        logical = os.cpu_count() or 1
    return {"model": model, "logical": logical, "physical": len(phys) or None}


def usable_cores():
    """logical CPUs this process may actually use: affinity mask, capped by a cgroup CPU quota when one is set"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = max(1, min(n, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = max(1, min(n, q // per))
        except Exception:
            pass
    return n


def bind_to_gpu_numa(index):
    """Pin this process (and so the first-touch placement of the page-locked buffers it allocates next) to the CPUs
    NVML reports as local to GPU `index` -- the multi-GPU e2e feed otherwise crosses the socket interconnect for half
    of the ranks (r1: 54 -> 39 GB/s per GPU at N = 8).  Returns the CPU list, or None when NVML has no answer."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = [64 * w + b for w, m in enumerate(mask) for b in range(64) if (int(m) >> b) & 1]
        allowed = os.sched_getaffinity(0)
        cpus = [c for c in cpus if c in allowed]
        if cpus:
            os.sched_setaffinity(0, cpus)
            return cpus
    except Exception:
        pass
    return None


def cpu_pool_rate(worker, make_args, units_per_worker, workers):
    """`workers` independent processes, one reference object each, disjoint inputs.  One untimed pass (process start,
    page-in, warm-up) and one timed pass; the rate is the AGGREGATE units / wall clock of the timed pass (all workers
    running concurrently, the number a user of all cores would see); the per-worker median and slowest times are
    reported beside it so that a straggler is visible instead of setting the number."""
    from oracle import ref_lib as R
    import multiprocessing as mp
    if not R.available():
        return None
    ctx = mp.get_context("spawn")
    with ctx.Pool(workers) as pool:
        t0 = time.perf_counter()
        pool.map(worker, [make_args(R.REF_PATH, 1234 + i, 1) for i in range(workers)])
        first = time.perf_counter() - t0
        t0 = time.perf_counter()
        times = pool.map(worker, [make_args(R.REF_PATH, 4321 + i, 0) for i in range(workers)])
        wall = time.perf_counter() - t0
    total = workers * units_per_worker
    return {"rate": total / wall, "rate_median_worker": total / float(np.median(times)), "rate_slowest_worker": total / max(times),
            "wall_s": wall, "worker_s_median": float(np.median(times)), "worker_s_max": float(max(times)), "first_wall_s": first}


def cpu_reference_rate(clips_per_worker, workers, warm=1):
    """The reference's own C path (oracle/_ref: built-in radix-2 FFT + naive double-accumulated dot; no
    FFTW/MKL/BLAS exist in this image) on `workers` independent processes, one object each, disjoint
    clips -- the fair all-cores figure, since the reference's OpenMP only splits frames inside a clip."""
    r = cpu_pool_rate(_cpu_worker, lambda path, seed, w: (path, seed, clips_per_worker, w), clips_per_worker * T, workers)
    if r is None:
        return None
    r["frames_per_s"] = r["rate"]
    return r


def _cpu_worker_cqt(args):
    lib_path, seed, clips, warm = args
    import ctypes
    sys.path.insert(0, ROOT)
    import audioflux_b200 as af
    from audioflux_b200 import capi
    lib = ctypes.CDLL(lib_path)
    capi.bind(lib)
    c = af.CQT(84, SR, _lib=lib)
    x = (0.1 * np.random.default_rng(seed).standard_normal((clips, L))).astype(np.float32)
    for i in range(warm):
        c.cqt_planes(x[i % clips])
    t0 = time.perf_counter()
    for i in range(clips):
        c.cqt_planes(x[i])
    return time.perf_counter() - t0


def _cpu_worker_cwt(args):
    lib_path, seed, clips, warm = args
    import ctypes
    sys.path.insert(0, ROOT)
    import audioflux_b200 as af
    from audioflux_b200 import capi
    lib = ctypes.CDLL(lib_path)
    capi.bind(lib)
    w = af.CWT(84, CWT_RADIX, SR, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False, _lib=lib)
    x = np.zeros((clips, 1 << CWT_RADIX), np.float32)
    x[:, :CWT_SAMPLES] = 0.1 * np.random.default_rng(seed).standard_normal((clips, CWT_SAMPLES))
    for i in range(warm):
        w.cwt_planes(x[i % clips])
    t0 = time.perf_counter()
    for i in range(clips):
        w.cwt_planes(x[i])
    return time.perf_counter() - t0


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = usable_cores()
    per = max(2, int(os.environ.get("AFB200_CPU_CLIPS_PER_WORKER", "16")))
    vals, runs = [], []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        r = cpu_reference_rate(per, cores)
        if r is None:
            emit({"impl": "reference", "unavailable": "oracle/_ref/libaudioflux_ref.so not built"})
            return 0
        vals.append(r["frames_per_s"])
        runs.append({k: r[k] for k in ("rate", "rate_median_worker", "rate_slowest_worker", "wall_s", "worker_s_median", "worker_s_max")})
    v = float(np.median(vals))
    frames_step = per * cores * T
    info = cpu_info()
    line = {
        "metric": "mfcc_frames_per_s", "value": v, "unit": "frames/s", "impl": "reference", "n_gpus": args.gpus,
        "steps": len(vals), "warmup": 1, "ms_per_step": 1e3 * frames_step / v, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the B200 arm's workload (same clips, same transform); each reference step is a bounded sample of it
        "config": {"workload": f"BASELINE config {'2' if args.gpus == 1 else '5-shaped'}: batch={args.batch} x 5 s 48 kHz clips per GPU, "
                               "STFT(2048,hop 512,hann)->mel128(slaney)->log10->DCT MFCC(40)",
                   "batch_per_gpu": args.batch, "clip_samples": L, "frames_per_clip": T,
                   "implementation": "reference CPU path: bftObj_bft(resultType=1) + xxccObj_xxcc of oracle/_ref (unmodified reference sources)",
                   "sample": f"{per} clips x {cores} worker processes per step ({per * cores} clips of the {args.batch}-clip batch shape)",
                   "cpu": info, "runs": runs},
        "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference",
                         "sample": f"{per * cores} clips ({frames_step} frames) per step, {cores} processes x 1 object, aggregate frames / wall "
                                   "of a steady pass (median over steps); reference built with gcc -O3, built-in radix-2 FFT + naive dot "
                                   "(no FFTW/MKL/BLAS in the image)", "cpu_model": info["model"], "physical_cores": info["physical"]},
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t_all,
    }
    emit(line)
    return 0


# --------------------------------------------------------------------------- BASELINE configs 3 (CQT) and 4 (CWT), N = 1
def _timed_ms(fn, steps, warm):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]


def bench_cqt_c3(dev, peaks, args, cores):
    """BASELINE config 3: batch = 1024 x 5 s clips, CQT 84 bins (12 per octave, fmin 32.7 Hz), device timed + e2e through
    cqtObj_cqtBatch with HOST pointers + parity gate (clip 0 and the last clip vs the numpy oracle)."""
    import torch
    import audioflux_b200 as af
    from audioflux_b200 import lib as L_
    from oracle import af_oracle as O
    lib = L_.get_lib()
    B = CQT_BATCH
    c = af.CQT(CQT_NUM, SR)
    Tq = c.cal_time_length(L)
    g = torch.Generator(device=dev).manual_seed(4321)
    x = 0.1 * torch.randn((B, L), generator=g, device=dev, dtype=torch.float32)
    re, im = c.cqt_batch(x)
    torch.cuda.synchronize()
    errs = []
    for i in (0, B - 1):
        wr, wi = O.cqt(x[i].cpu().numpy(), CQT_NUM, SR, norm=O.NORM_AREA)
        want = wr + 1j * wi
        got = re[i].cpu().numpy() + 1j * im[i].cpu().numpy()
        errs.append(float(np.abs(got - want).max() / np.abs(want).max()))
    if not max(errs) < 1e-4:
        return {"error": f"CQT parity gate failed: rel err {errs}"}
    del re, im
    n0 = lib.afb200_kernelLaunchCount()
    ms = _timed_ms(lambda: c.cqt_batch(x), steps=args.steps, warm=3)
    launches = (lib.afb200_kernelLaunchCount() - n0) // (len(ms) + 3)
    ms_step = float(np.mean(ms))
    # end to end: the C-ABI call with page-locked HOST buffers (chunked copy-in / transform / copy-out inside)
    xh = torch.empty((B, L), dtype=torch.float32).pin_memory()
    xh.copy_(x.cpu())
    del x
    xh_np = xh.numpy()
    rh = torch.empty((B, Tq, CQT_NUM), dtype=torch.float32).pin_memory()
    ih = torch.empty((B, Tq, CQT_NUM), dtype=torch.float32).pin_memory()
    import ctypes as C
    fn = lib.cqtObj_cqtBatch

    def e2e():
        L_.check(fn(c._obj, C.c_void_p(xh_np.ctypes.data), L, B, C.c_void_p(rh.numpy().ctypes.data),
                    C.c_void_p(ih.numpy().ctypes.data), 0, None), "cqtObj_cqtBatch(host)")
    e2e()
    t0 = time.perf_counter()
    n_e = 3
    for _ in range(n_e):
        e2e()
    e2e_s = (time.perf_counter() - t0) / n_e
    bytes_clip = 4 * L + 2 * 4 * Tq * CQT_NUM                       # compulsory: samples in, two planes out
    achieved = B * bytes_clip / (ms_step * 1e-3) / 1e9
    out = {"metric": "cqt_clips_per_s", "value": B / (ms_step * 1e-3), "unit": "clips/s", "ms_per_step": ms_step,
           "per_step_ms": ms, "frames_per_s": B * Tq / (ms_step * 1e-3),
           "config": {"workload": f"BASELINE config 3: batch={B} x 5 s 48 kHz clips, CQT {CQT_NUM} bins (12/octave, fmin 32.7 Hz, hann, hop {c.slide_length})",
                      "frames_per_clip": Tq, "parity_rel_err_clip0_last": errs},
           "e2e": {"value": B / e2e_s, "unit": "clips/s", "h2d_bytes_per_step": B * L * 4, "d2h_bytes_per_step": 2 * B * Tq * CQT_NUM * 4},
           "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                        "traffic": None, "algorithmic_bytes_per_step": B * bytes_clip,
                        "fp32_tflops": B * 7 * Tq * 512 * 24 * 2 / (ms_step * 1e-3) / 1e12,
                        "note": "FP32-FMA bound (7 octaves x T x 512 taps x 24 real MACs per frame), not HBM bound"}}
    if not args.no_cpu_baseline:
        per = 2
        r = cpu_pool_rate(_cpu_worker_cqt, lambda path, seed, w: (path, seed, per, w), per, cores)
        if r:
            out["cpu_baseline"] = {"value": r["rate"], "unit": "clips/s", "cores": cores, "kind": "reference",
                                   "sample": f"{cores} processes x {per} clips of 5 s, cqtObj_cqt of oracle/_ref, aggregate clips / wall",
                                   "worker_s_median": r["worker_s_median"], "worker_s_max": r["worker_s_max"]}
    return out


def bench_cwt_c4(dev, peaks, args, cores):
    """BASELINE config 4: batch = 512 x 10 s clips (480 000 samples zero-padded to 2^19), CWT morlet 84 scales.  The two
    output planes are 352 MB per clip (180 GB for the batch): the batch runs in chunks whose planes reuse one device
    buffer (a consumer would reduce them in place); e2e copies every chunk's planes to page-locked host memory."""
    import torch
    import audioflux_b200 as af
    from audioflux_b200 import lib as L_
    from oracle import af_oracle as O
    import ctypes as C
    lib = L_.get_lib()
    B, N, chunk = CWT_BATCH, 1 << CWT_RADIX, int(os.environ.get("AFB200_CWT_CHUNK", "16"))
    w = af.CWT(CWT_NUM, CWT_RADIX, SR, wavelet_type=af.WaveletContinueType.MORLET, is_padding=False)
    g = torch.Generator(device=dev).manual_seed(977)
    x = torch.zeros((B, N), device=dev, dtype=torch.float32)
    x[:, :CWT_SAMPLES] = 0.1 * torch.randn((B, CWT_SAMPLES), generator=g, device=dev, dtype=torch.float32)
    re = torch.empty((chunk, CWT_NUM, N), device=dev, dtype=torch.float32)
    im = torch.empty_like(re)
    fn = lib.cwtObj_cwtBatch
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def run_chunk(c0):
        nb = min(chunk, B - c0)
        L_.check(fn(w._obj, C.c_void_p(x[c0].data_ptr()), nb, C.c_void_p(re.data_ptr()), C.c_void_p(im.data_ptr()), 1, stream), "cwtObj_cwtBatch")

    def step():
        for c0 in range(0, B, chunk):
            run_chunk(c0)
    # parity gate: the LAST clip of the last chunk vs the numpy oracle
    run_chunk(B - chunk)
    torch.cuda.synchronize()
    wr, wi = O.cwt(x[B - 1].cpu().numpy(), CWT_NUM, CWT_RADIX, SR, wavelet=O.WAVE_MORLET, is_pad=False)
    got = re[chunk - 1].cpu().numpy() + 1j * im[chunk - 1].cpu().numpy()
    want = wr + 1j * wi
    err = float(np.abs(got - want).max() / np.abs(want).max())
    del wr, wi, got, want
    if not err < 1e-4:
        return {"error": f"CWT parity gate failed: rel err {err}"}
    n0 = lib.afb200_kernelLaunchCount()
    ms = _timed_ms(step, steps=args.steps, warm=1)
    launches = (lib.afb200_kernelLaunchCount() - n0) // (len(ms) + 1)
    ms_step = float(np.mean(ms))
    # end to end: cwtObj_cwtBatch with HOST pointers, chunk by chunk (inputs from and planes to page-locked host memory)
    xh = torch.empty((chunk, N), dtype=torch.float32).pin_memory()
    xh.copy_(x[:chunk].cpu())
    rh = torch.empty((chunk, CWT_NUM, N), dtype=torch.float32).pin_memory()
    ih = torch.empty((chunk, CWT_NUM, N), dtype=torch.float32).pin_memory()
    xp, rp, ip = xh.numpy().ctypes.data, rh.numpy().ctypes.data, ih.numpy().ctypes.data

    def e2e_chunk():
        L_.check(fn(w._obj, C.c_void_p(xp), chunk, C.c_void_p(rp), C.c_void_p(ip), 0, None), "cwtObj_cwtBatch(host)")
    e2e_chunk()
    n_chunks = int(os.environ.get("AFB200_CWT_E2E_CHUNKS", "8"))      # bounded sample of the 32 chunks of one step
    t0 = time.perf_counter()
    for _ in range(n_chunks):
        e2e_chunk()
    e2e_s_per_clip = (time.perf_counter() - t0) / (n_chunks * chunk)
    bytes_clip = 4 * CWT_SAMPLES + 2 * 4 * CWT_NUM * N
    achieved = B * bytes_clip / (ms_step * 1e-3) / 1e9
    # DRAM bytes of the dominant kernel (k_cwt_fused_w) from the committed ncu capture: tools/cwt_prof.py transforms 4 clips per
    # launch, the bench chunk-size clips -- the kernel walks (clip, scale) items in groups of 4, so its traffic scales with the clips
    cwt_summary, cwt_capture_clips = "r2_final_cwt_ncu.txt", 4
    t4 = ncu_traffic(cwt_summary)
    cwt_traffic = int(t4 / cwt_capture_clips * chunk) if t4 else None
    out = {"metric": "cwt_clips_per_s", "value": B / (ms_step * 1e-3), "unit": "clips/s", "ms_per_step": ms_step, "per_step_ms": ms,
           "config": {"workload": f"BASELINE config 4: batch={B} x 10 s 48 kHz clips (480000 samples zero-padded to 2^19), CWT morlet {CWT_NUM} scales (octave)",
                      "chunk_clips": chunk, "output": "two planes of 352 MB per clip; each chunk's planes overwrite one device buffer",
                      "parity_rel_err_last_clip": err},
           "e2e": {"value": 1.0 / e2e_s_per_clip, "unit": "clips/s", "h2d_bytes_per_step": B * N * 4, "d2h_bytes_per_step": 2 * B * CWT_NUM * N * 4,
                   "sample": f"{n_chunks} of the {B // chunk} chunks of a step, each through cwtObj_cwtBatch with HOST pointers"},
           "gpu_launches": int(launches),
           "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                        "traffic": cwt_traffic, "traffic_source": f"profiles/{cwt_summary} ({cwt_capture_clips} clips per launch) scaled to the bench's {chunk}-clip launches" if cwt_traffic else None,
                        "kernel": "k_cwt_fused_w", "algorithmic_bytes_per_launch": chunk * bytes_clip,
                        "algorithmic_bytes_per_step": B * bytes_clip}}
    del x, re, im
    if not args.no_cpu_baseline:
        workers = max(1, min(cores, 32))                            # 0.6 GB per worker (bank table + planes at N = 2^19)
        r = cpu_pool_rate(_cpu_worker_cwt, lambda path, seed, w_: (path, seed, 1, 0), 1, workers)
        if r:
            out["cpu_baseline"] = {"value": r["rate"], "unit": "clips/s", "cores": workers, "kind": "reference",
                                   "sample": f"{workers} processes x 1 clip of 2^19 samples, cwtObj_cwt of oracle/_ref, aggregate clips / wall (two passes, second timed)",
                                   "worker_s_median": r["worker_s_median"], "worker_s_max": r["worker_s_max"]}
    return out


# --------------------------------------------------------------------------- B200 arm
def run_b200_arm(args):
    import torch
    import audioflux_b200 as af
    from audioflux_b200 import lib as L_

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist_
        dist = dist_
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line, but NCCL prints "NCCL version ..." there when the box sets NCCL_DEBUG:
        # from here on file descriptor 1 is stderr, and the JSON line is written to the saved real stdout (emit())
        global _REAL_STDOUT
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    lib = L_.get_lib()

    B = args.batch
    S, D = af.SpectralFilterBankScaleType, af.SpectralDataType
    bft = af.BFT(NMEL, RADIX, SR, slide_length=HOP, scale_type=S.MEL, data_type=D.POWER)
    g = torch.Generator(device=dev).manual_seed(1234 + 2 + rank)
    x = 0.1 * torch.randn((B, L), generator=g, device=dev, dtype=torch.float32)
    # N > 1: the gather of the per-rank results.  Default "peer": ONE kernel per step, whose epilogue stores every
    # finished tile into all ranks' gathered arrays over NVLink (audioflux_b200/dist.py:PeerScatter), then a 4-byte
    # all-reduce as the cross-rank fence.  Fallback / comparison "nccl": chunked compute with chunk k's
    # all_gather_into_tensor on a side stream while chunk k+1 computes (OverlappedGather).
    overlap = scatter = None
    gather_mode = "none"
    if world > 1:
        from audioflux_b200.dist import OverlappedGather, PeerScatter
        gather_mode = args.gather
        if gather_mode == "peer":
            try:
                scatter = PeerScatter(bft, B, L, NCC)
            except RuntimeError as e:
                if rank == 0:
                    print(f"[bench] peer scatter unavailable, using NCCL all-gather: {e}", file=sys.stderr)
                gather_mode = "nccl"
        if gather_mode == "nccl":
            overlap = OverlappedGather(chunks=args.gather_chunks)

    def step(inp=None):
        inp = x if inp is None else inp
        if scatter is not None:
            out = scatter(inp)
            scatter.fence()
            return out
        if overlap is not None:
            return overlap(lambda c: bft.mfcc_batch(c, NCC), inp)
        return bft.mfcc_batch(inp, NCC)

    # parity gate on this very configuration before any timing counts (clip 0 vs the numpy oracle)
    parity = None
    if rank == 0:
        from oracle import af_oracle as O
        out = bft.mfcc_batch(x, NCC)          # no collective here: only rank 0 runs the gate
        torch.cuda.synchronize()
        want = O.mfcc(x[0].cpu().numpy(), SR, RADIX, HOP, NMEL, NCC)
        parity = float(np.abs(out[0].cpu().numpy() - want).max() / np.abs(want).max())
        if not parity < 1e-4:
            emit({"error": f"parity gate failed: rel err {parity}"})
            return 1

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    # gather gate (N > 1): rank 0 regenerates the LAST rank's seeded shard, transforms it locally and compares with
    # what arrived in its gathered array -- bit for bit (results do not depend on which GPU computed them)
    gather_ok = None
    if world > 1 and rank == 0:
        gl = torch.Generator(device=dev).manual_seed(1234 + 2 + (world - 1))
        xl = 0.1 * torch.randn((B, L), generator=gl, device=dev, dtype=torch.float32)
        want_l = bft.mfcc_batch(xl[:8], NCC)
        res = step()
        torch.cuda.synchronize()
        got_l = res[world - 1][:8] if scatter is not None else res[0][(world - 1) * res[0].shape[0] // world:][:8]
        gather_ok = bool(torch.equal(got_l, want_l))
        del xl
    elif world > 1:
        step()
        torch.cuda.synchronize()
    if dist:
        dist.barrier()
    if gather_ok is False:
        emit({"error": "gather gate failed: the last rank's block did not arrive intact on rank 0"})
        return 1

    launches0 = lib.afb200_kernelLaunchCount()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    kern_ms = []
    torch.cuda.synchronize()
    sampler.mark(True)
    ev[0].record()
    for i in range(args.steps):
        last = step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    sampler.mark(False)
    if args.dump_outputs and rank == 0:
        if scatter is not None:            # (world, B, T, cc)
            last = last.reshape(world * B, T, NCC)
        elif overlap is not None:          # chunk k gathered as (world * B / chunks, T, cc), rank-major inside the chunk
            last = torch.cat([o.view(world, -1, T, NCC) for o in last], dim=1).reshape(world * B, T, NCC)
        dump_outputs(args.dump_outputs, {"mfcc": last})
    if dist:
        dist.barrier()
    launches = lib.afb200_kernelLaunchCount() - launches0
    clocks = sampler.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    if world > 1:                      # kernel-only duration for the roofline: one untimed-by-the-metric extra pass
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        for _ in range(3):
            bft.mfcc_batch(x, NCC)
        k1.record()
        torch.cuda.synchronize()
        kernel_ms = k0.elapsed_time(k1) / 3
    else:
        kernel_ms = float(np.mean(per_step))
    t = torch.tensor([total_ms], device=dev)
    if dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_step = total_ms / args.steps
    value = world * B * T / (ms_step * 1e-3)

    # ---- end to end through the public API with HOST buffers (pinned), H2D + D2H inside the timed region
    xh = torch.empty((B, L), dtype=torch.float32).pin_memory()
    xh.copy_(x.cpu())
    oh = torch.empty((B, T, NCC), dtype=torch.float32).pin_memory()
    xd = torch.empty_like(x)

    xh_np, oh_np = xh.numpy(), oh.numpy()           # views of the page-locked buffers for the C-ABI host-pointer call
    h2d_stream = torch.cuda.Stream()
    h2d_done = [torch.cuda.Event() for _ in range(8)]

    def e2e_step():
        if world == 1:
            # the call a user of the C ABI makes: bftObj_mfccBatch with HOST pointers (memKind 0); inside, the library
            # pipelines copy-in / transform / copy-out over chunks and returns when `oh` is complete
            bft.mfcc_batch(xh_np, NCC, out=oh_np)
            return
        if scatter is not None:
            # stream the shard in chunk by chunk: copy-in of chunk k+1 on a side stream overlaps the fused transform +
            # scatter of chunk k; then the cross-rank fence and this rank's own slot of the gathered array -> host
            cur = torch.cuda.current_stream()
            nchunk = 8
            per = (B + nchunk - 1) // nchunk
            for k in range(nchunk):
                lo, hi = k * per, min(B, (k + 1) * per)
                if lo >= hi:
                    break
                with torch.cuda.stream(h2d_stream):
                    if k == 0:
                        h2d_stream.wait_stream(cur)                  # xd is free again (previous step's kernels done)
                    xd[lo:hi].copy_(xh[lo:hi], non_blocking=True)
                    h2d_done[k].record(h2d_stream)
                cur.wait_event(h2d_done[k])
                scatter(xd[lo:hi], clip_offset=lo)
            scatter.fence()
            oh.copy_(scatter.gathered[rank], non_blocking=True)
            return
        xd.copy_(xh, non_blocking=True)            # --gather nccl: copy-in, chunked compute + overlapped all-gather
        res = step(xd)
        per = res[0].shape[0] // world
        for k, o in enumerate(res):                # this rank's own rows of every gathered chunk -> host
            oh[k * per:(k + 1) * per].copy_(o[rank * per:(rank + 1) * per], non_blocking=True)

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_e2e = args.steps
    e0.record()
    for _ in range(n_e2e):
        e2e_step()
    e1.record()
    torch.cuda.synchronize()
    te = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if dist:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * B * T / (float(te.item()) / n_e2e * 1e-3)

    if scatter is not None:
        torch.cuda.synchronize()
        dist.barrier()                 # nobody unmaps while a peer may still be storing
        scatter.close()
    if rank != 0:
        if dist:
            dist.destroy_process_group()
        return 0

    peaks, peak_kind = measured_peaks()
    achieved = B * BYTES_PER_CLIP / (kernel_ms * 1e-3) / 1e9
    cores = usable_cores()
    per_cpu = max(2, int(os.environ.get("AFB200_CPU_CLIPS_PER_WORKER", "16")))
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_rate(per_cpu, cores)
    kernel_name = "k_mfcc_fused<5,0>" if os.environ.get("AFB200_MFCC_KERNEL") == "v1" else "k_mfcc_fused2<5>"
    summary = os.environ.get("AFB200_NCU_SUMMARY", "r1_final_mfcc_fused_ncu_summary.txt" if "fused<" in kernel_name
                             else "r2_final_mfcc_fused2_ncu_summary.txt")
    traffic = ncu_traffic(summary) if (B == 1024 and L == 240000) else None
    if traffic is None and "fused2" in kernel_name and B == 1024 and L == 240000:
        summary = "r2_mfcc_fused2_ncu_summary.txt"                   # the capture at the start of the round
        traffic = ncu_traffic(summary)
    line = {
        "metric": "mfcc_frames_per_s", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"BASELINE config {'2' if world == 1 else '5-shaped'}: batch={B} x 5 s 48 kHz clips per GPU, "
                               "STFT(2048,hop 512,hann)->mel128(slaney)->log10->DCT MFCC(40), fused kernel",
                   "batch_per_gpu": B, "clip_samples": L, "frames_per_clip": T,
                   "l2": "inputs (983 MB per GPU) exceed the 126 MB L2; no explicit flush needed",
                   "collective": {"none": "none",
                                  "peer": "fused: the kernel epilogue stores each tile into every rank's gathered (world,B,T,40) array "
                                          "over NVLink P2P (cudaIpc-mapped), then a 4-byte NCCL all-reduce as the cross-rank fence",
                                  "nccl": f"nccl all_gather of (B,T,40) per step in {args.gather_chunks} chunks overlapped with compute"}[gather_mode],
                   "gather_gate_bitexact": gather_ok,
                   "host_binding": (f"rank pinned to the {len(numa_cpus)} CPUs local to its GPU (NVML affinity) before allocating page-locked buffers"
                                    if numa_cpus else "none"),
                   "parity_rel_err_clip0": parity},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": B * L * 4, "d2h_bytes_per_step": B * T * NCC * 4,
                "steps": n_e2e},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                     "frac": achieved / peaks["hbm_gbs"],
                     # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of this kernel at this configuration, parsed at
                     # run time from the committed ncu --set full summary under profiles/ (None if that file is absent)
                     "traffic": traffic, "traffic_source": f"profiles/{summary}" if traffic else None, "peak_kind": peak_kind,
                     "kernel": kernel_name, "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": B * BYTES_PER_CLIP,
                     "frame_read_model_frac": (B * T * BYTES_PER_FRAME_READ_MODEL / (kernel_ms * 1e-3) / 1e9) / peaks["hbm_gbs"],
                     "fp32_tflops": B * T * FLOP_PER_FRAME / (kernel_ms * 1e-3) / 1e12},
        "per_step_ms": per_step,
    }
    if cpu:
        info = cpu_info()
        line["cpu_baseline"] = {"value": cpu["frames_per_s"], "unit": "frames/s", "cores": cores, "kind": "reference",
                                "sample": f"{cores} processes x {per_cpu} clips, aggregate frames / wall of a steady pass, "
                                          "oracle/_ref (gcc -O3, built-in radix-2 FFT + naive dot)",
                                "rate_median_worker": cpu["rate_median_worker"], "rate_slowest_worker": cpu["rate_slowest_worker"],
                                "cpu_model": info["model"], "physical_cores": info["physical"]}
    if world == 1 and not args.no_extra:
        # BASELINE configs 3 and 4 on the same line (their own value / e2e / roofline / cpu_baseline / parity gate)
        del x, xd, xh, oh
        torch.cuda.empty_cache()
        for key, fn in (("cqt", bench_cqt_c3), ("cwt", bench_cwt_c4)):
            try:
                line[key] = fn(dev, peaks, args, cores)
            except Exception as exc:                                # the headline line must survive a failure here
                line[key] = {"error": f"{type(exc).__name__}: {exc}"}
            torch.cuda.empty_cache()
    emit(line)
    if dist:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH_PER_GPU, help="clips per GPU (default: BASELINE config 2)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the CQT (config 3) / CWT (config 4) keys")
    ap.add_argument("--gather-chunks", type=int, default=4, help="N>1, --gather nccl: chunks per step for compute/all-gather overlap")
    ap.add_argument("--gather", choices=("peer", "nccl"), default="peer",
                    help="N>1: 'peer' = all-gather fused into the kernel epilogue (NVLink P2P stores); 'nccl' = overlapped NCCL all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the MFCCs of the last one -- the headline path; the CQT / CWT keys "
                         "dump nothing -- to DIR/mfcc.npy (float32; a fixed sample of clips when the batch exceeds 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the B200 path's MFCCs; it does not apply to --impl reference")
        return run_reference_arm(args)
    return run_b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
