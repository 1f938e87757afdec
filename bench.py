#!/usr/bin/env python
"""bench.py — DAB transmission frames/s through the full B200 decode chain (driver contract).

    python bench.py --gpus N --steps K --warmup W           # our arm (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own CPU path on the host cores

A "step" = one pass of the hot path over one batch: every one of the `--batch` independent ensemble streams of a rank
decodes its next 96 ms transmission frame (time sync -> 76 FFTs + DQPSK demap -> FIC Viterbi + CRC -> one 96 kbit/s
EEP-3A DAB+ sub-channel: time de-interleave, Viterbi, energy dispersal, RS(120,110) + Fire code + AU CRC).
Workload = BASELINE.json configs[3]/[4]: batch = 8192 frames per GPU, streams sharded across ranks with no data-path
collective (weak scaling); a one-int32 NCCL broadcast of the work descriptor is the only communication.

value    whole-job frames/s with the IQ already resident in HBM (CUDA events on the library's stream, max over ranks)
e2e      the same through dabb_process() with HOST (pinned) IQ buffers: H2D of every step's samples and D2H of the
         results inside the timed region
roofline dominant kernel (ofdm_demod_kernel) timed alone with CUDA events: algorithmic bytes / duration vs the
         measured HBM copy bandwidth in MEASURED_PEAKS.json
cpu_baseline  the unmodified reference backend (oracle/_ref, KISS-FFT build) on the host cores, bounded sample
"""
import argparse
import importlib.util
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
TF, TU, TS, TNULL = 196608, 2048, 2552, 2656
RING_FRAMES = 5
BUF_LEN = (RING_FRAMES + 1) * TF + 4096
BITRATE, SUBCH_CU = 96, 72
# bytes one frame must move through the OFDM kernel: PRS (2048) + 75 symbols x 2552 samples read once, 75 x 3072 softbits written
OFDM_BYTES_PER_FRAME = (TU + 75 * TS) * 8 + 75 * 3072
SURVEY_BYTES_PER_FRAME = 1803264   # SURVEY.md §8(d): also counts the null symbol, which this kernel never reads
ACS_PER_FRAME = (4 * 774 + 4 * 2310) * 64


def _baseline_metric():
    # BASELINE.json's own wording of the metric, so that the driver can match the line to it
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "DAB transmission frames/sec (96 ms, 2.048 Msps IQ) at 1/2/4/8 B200 vs ref CPU"


METRIC = _baseline_metric()


def load_pkg():
    d = os.path.join(ROOT, "welle.io_b200")
    if "welle_io_b200" in sys.modules:
        return sys.modules["welle_io_b200"]
    spec = importlib.util.spec_from_file_location("welle_io_b200", os.path.join(d, "__init__.py"), submodule_search_locations=[d])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["welle_io_b200"] = mod
    spec.loader.exec_module(mod)
    return mod


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML, ~2 ms per sample)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz, self.err = index, [], set(), False, None, None
        self.ready = threading.Event()       # set once NVML is initialised (that can take longer than the whole timed region on a fresh box)
        self.armed = False                   # samples count only while the timed region runs

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                     "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
            self.ready.set()
            while not self.stop_flag:
                if self.armed:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    for k, bit in names.items():
                        if r & bit:
                            self.reasons.add(k)
                time.sleep(0.002)
        except Exception as e:  # noqa
            self.err = repr(e)
            self.ready.set()

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples), "error": self.err}


def log(msg):
    print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


# ------------------------------------------------------------------------------------------------ reference arm
def _ref_worker(args):
    n_frames, seed = args
    import dabtx
    from oracle.bind import Ref
    r = Ref()
    tx = dabtx.DabTx(seed=seed)
    iq = tx.frames(n_frames)
    e = r.e2e(iq, disable_coarse=True, select_at_fib=24, dump_path=f"/tmp/bench_ref_{os.getpid()}.msc")
    # seconds = wall time from RadioReceiver::restart until the input was exhausted (teardown/drain waits excluded)
    return e["frames_done"], float(e["seconds"]), int(e["fibs"][:, 0].sum()), len(e["fibs"])


def run_reference_cpu(n_procs, frames_per_proc):
    """the reference's own RadioReceiver (3+ threads per stream) on `n_procs` concurrent streams; frames/s = decoded frames / wall time"""
    ctx = mp.get_context("fork")
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(2); os.dup2(devnull, 2)      # the reference logs to stderr
    try:
        t0 = time.time()
        with ctx.Pool(n_procs) as pool:
            out = pool.map(_ref_worker, [(frames_per_proc, 0x1000 + i) for i in range(n_procs)])
        wall = time.time() - t0
    finally:
        os.dup2(saved, 2); os.close(devnull)
    frames = sum(o[0] for o in out)
    busy = max(o[1] for o in out)
    return frames / busy, frames, busy, wall, sum(o[2] for o in out), sum(o[3] for o in out)


def reference_stage_level():
    """SURVEY 8(d) CPU timing (i): the reference's own stage functions, single thread, on a few synthetic frames: one frame's
    OFDM demod (PRS + 75 data symbols: fft::Forward + demap loop), FIC (processFicBlock: 4 Viterbi + CRC), MSC (4 x EEPProtection::
    deconvolve + dedisperse) and RSDecoder::DecodeSuperframe; seconds per frame and frames/s on one core"""
    import dabtx
    from oracle.bind import Ref
    r = Ref()
    tx = dabtx.DabTx(seed=0x77)
    iq = tx.frames(4)
    st = 2 * TF + TNULL + 504
    prs, syms = iq[st: st + 2048], iq[st + 2048: st + 2048 + 75 * 2552]
    sf = tx.superframes[0] if tx.superframes else None
    reps = 5
    t0 = time.perf_counter()
    for _ in range(reps):
        soft = r.demod_frame(prs, syms)
    t_ofdm = (time.perf_counter() - t0) / reps
    fic = np.ascontiguousarray(soft[:3].reshape(-1))
    t0 = time.perf_counter()
    for _ in range(reps):
        r.fic_decode(fic)
    t_fic = (time.perf_counter() - t0) / reps
    cif = np.ascontiguousarray(soft[3:21].reshape(-1)[:SUBCH_CU * 64])
    t0 = time.perf_counter()
    for _ in range(reps):
        for _c in range(4):
            r.eep_deconvolve(BITRATE, 1, 3, cif, True)
    t_msc = (time.perf_counter() - t0) / reps
    t_rs = 0.0
    if sf is not None:
        t0 = time.perf_counter()
        for _ in range(reps * 4):
            r.rs_decode_superframe(sf)
        t_rs = (time.perf_counter() - t0) / (reps * 4) * 0.8       # 4 superframes per 5 transmission frames
    tot = t_ofdm + t_fic + t_msc + t_rs
    return {"seconds_per_frame": {"ofdm_demod": t_ofdm, "fic": t_fic, "msc_96k_eep3a": t_msc, "rs_superframe": t_rs}, "frames_per_s_one_core": 1.0 / tot,
            "note": "unmodified reference stage functions called in a single-threaded loop (ctypes call overhead included, < 1 %)"}


def _stage_worker(args):
    """one process: the reference's stage functions over `seconds` of wall time on its own synthetic frames; returns frames done"""
    seed, seconds = args
    import dabtx
    from oracle.bind import Ref
    r = Ref()
    tx = dabtx.DabTx(seed=seed)
    iq = tx.frames(4)
    st = 2 * TF + TNULL + 504
    prs, syms = iq[st: st + 2048], iq[st + 2048: st + 2048 + 75 * 2552]
    sf = tx.superframes[0] if tx.superframes else None
    done, k = 0, 0
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        soft = r.demod_frame(prs, syms)
        r.fic_decode(np.ascontiguousarray(soft[:3].reshape(-1)))
        cif = np.ascontiguousarray(soft[3:21].reshape(-1)[:SUBCH_CU * 64])
        for _c in range(4):
            r.eep_deconvolve(BITRATE, 1, 3, cif, True)
        k += 1
        if sf is not None and k % 5 != 0:          # 4 superframes per 5 transmission frames
            r.rs_decode_superframe(sf)
        done += 1
    return done, time.perf_counter() - t0


def reference_stage_level_all_cores(n_procs, seconds=8.0):
    """SURVEY 8(d) CPU timing (i), second half: the same unmodified reference stage functions (fft::Forward + demap loop, processFicBlock,
    EEPProtection::deconvolve, RSDecoder::DecodeSuperframe) in n_procs processes over disjoint frames - an upper bound for what the
    reference's kernels can do on this host (no time sync, no oscillator, no thread hand-over)"""
    ctx = mp.get_context("fork")
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(2); os.dup2(devnull, 2)
    try:
        with ctx.Pool(n_procs) as pool:
            out = pool.map(_stage_worker, [(0x2000 + i, seconds) for i in range(n_procs)])
    finally:
        os.dup2(saved, 2); os.close(devnull)
    frames = sum(o[0] for o in out); busy = max(o[1] for o in out)
    return {"value": frames / busy, "unit": "frames/s", "processes": n_procs, "frames": frames, "seconds": busy,
            "note": "unmodified reference stage functions (OFDM demod of 76 symbols, FIC, 4 x MSC 96 kbit/s EEP-3A, RS) in a loop, one process per core over disjoint frames"}


def effective_cores():
    """cores this process may really use: affinity mask and the cgroup CPU quota (a container can see 128 cores and own a dozen)"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    return {"visible": os.cpu_count() or 1, "affinity": n, "cgroup_quota": quota, "effective": min(n, quota) if quota else n}


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.bind import Ref
    if not Ref.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libwelle_ref.so missing (built only where /root/reference exists)"}))
        return
    cores = max(1, int(effective_cores()["effective"]))
    n_procs = max(1, min(cores // 3, 48))       # one reference receiver runs ~3 busy threads (OFDM, decoder, DabAudio)
    vals = []
    for it in range(a.warmup + a.steps):
        v, frames, busy, wall, ok, tot = run_reference_cpu(n_procs, a.ref_frames)
        if it >= a.warmup:
            vals.append((v, busy))
    v = float(np.mean([x[0] for x in vals]))
    ms = float(np.mean([x[1] for x in vals]) * 1e3)
    sample = f"{n_procs} concurrent reference RadioReceiver instances x {a.ref_frames} synthetic frames each (FIC + one 96 kbit/s EEP-3A DAB+ sub-channel), KISS-FFT build"
    try:
        stage_all = reference_stage_level_all_cores(cores)
    except Exception as e:  # noqa
        stage_all = {"error": repr(e)}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+int", "data": "synthetic",
            "config": config_dict(a, None),
            "cpu_baseline": {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference", "sample": sample, "cores_detail": effective_cores(),
                             "stage_level_all_cores": stage_all,
                             "note": "value = the stock code path (RadioReceiver with its own threads, flow-controlled memory input); stage_level_all_cores = the reference's stage functions alone on every core, the most the reference's kernels can give on this host"},
            "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def config_dict(a, groups):
    return {"workload": f"batch={a.batch} independent Mode-I ensembles per GPU, 1 transmission frame per stream per step: full chain sync+76xFFT+DQPSK -> FIC Viterbi+CRC -> 96 kbit/s EEP-3A DAB+ sub-channel (time de-interleave, Viterbi, RS(120,110)+Fire code) [BASELINE.json configs[3]/[4]]",
            "batch_frames_per_gpu": a.batch, "subchannel": "96 kbit/s EEP 3-A, 72 CU, DAB+", "snr_db": a.snr, "fft_mode": "exact(KISS-bit-identical)" if a.fft_mode == 0 else "fma",
            "parallelism": f"streams sharded over {a.gpus} GPU(s), no data-path collective", "l2_policy": "inputs (12.9 GB/step at batch 8192) far exceed the 126 MB L2; no flush needed",
            "carrier_offset": "0 Hz (headline): fine corrector stays 0 and the oscillator multiply is skipped; roofline.oscillator_active repeats the run with an offset",
            "input": "8 distinct 5-frame periodic rings (different seeds) replicated over the batch + per-stream AWGN; the timed region is steps x ~4.7 ms",
            "ofdm_tail_split": "last resident/2 frames of the launch as 5 CTAs of 15 symbols" if not getattr(a, "no_tail_split", False) else "off",
            "nco_mode": "exact (headline; oscillator_active reports exact and fast)",
            "ofdm_groups": groups}


# ------------------------------------------------------------------------------------------------ our arm
def make_rings(n_distinct):
    import dabtx
    rings = []
    for i in range(n_distinct):
        _, ring = dabtx.periodic_ring(0xB200 + i, RING_FRAMES)
        rings.append(ring)
    return np.stack(rings)


def prefer_host_memory_near_gpu(index):
    """Host allocations of this rank (the pinned IQ ring of the e2e leg) should come from the NUMA node its GPU hangs off: what
    `numactl --preferred` per rank does, through set_mempolicy(MPOL_PREFERRED).  Returns what was done (goes into `config`)."""
    info = {"gpu_numa_node": None, "policy": "default"}
    try:
        import ctypes
        import pynvml as nv
        nv.nvmlInit()
        bus = nv.nvmlDeviceGetPciInfo(nv.nvmlDeviceGetHandleByIndex(index)).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node = -1
        for cand in (bus.lower(), bus.lower()[4:] if len(bus) > 12 else bus.lower()):
            pth = f"/sys/bus/pci/devices/{cand}/numa_node"
            if os.path.exists(pth):
                node = int(open(pth).read().strip()); break
        info["gpu_numa_node"] = node
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if node >= 0 and len(nodes) > 1:
            mask = ctypes.c_ulong(1 << node)
            libc = ctypes.CDLL(None, use_errno=True)
            rc = libc.syscall(238, 1, ctypes.byref(mask), 8 * ctypes.sizeof(mask))       # x86-64 SYS_set_mempolicy, MPOL_PREFERRED
            info["policy"] = f"preferred node {node}" if rc == 0 else f"set_mempolicy failed (errno {ctypes.get_errno()})"
    except Exception as e:  # noqa
        info["policy"] = "default (" + type(e).__name__ + ")"
    return info


DUMP_STREAMS = 1024      # streams of the batch (a fixed, seeded sample) whose outputs --dump-outputs writes


def dump_outputs(out_dir, a, pkg, device, S, buf, n_calls, buf_start_for):
    """--dump-outputs: the outputs of the last timed step, one float64 .npy per array.  dabb_process_async hands nothing back to its
    caller, so a second context with the timed one's configuration repeats the same n_calls steps on the same input and takes the last
    one through dabb_process (= dabb_process_async + the copies of the step's outputs to the host).  Written for a seeded sample of
    DUMP_STREAMS streams (streams.npy): every field of the per-stream results, the FIBs, and the sub-channel's logical frames (msc) and
    superframe (sf)."""
    c = pkg.Context(n_streams=S, device=device, fft_mode=a.fft_mode, disable_coarse=True, n_subch_slots=1, max_subch_cu=SUBCH_CU,
                    ofdm_tail_split=-1 if a.no_tail_split else 0)
    c.select_subchannel(0, SUBCH_CU, BITRATE, eep_profile_a=True, eep_level=3, dabplus=True)
    for call in range(n_calls - 1):
        c.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(call), BUF_LEN)
    out = c.process(buf, BUF_LEN, buf_start_for(n_calls - 1), BUF_LEN, msc_stride=3 * BITRATE, sf_stride=15 * BITRATE)
    c.close()
    pick = np.sort(np.random.default_rng(0xD0D0).choice(S, min(S, DUMP_STREAMS), replace=False))
    r = out["results"][pick]
    arrays = {"streams": pick, "fibs": out["fibs"][pick], "msc": out["msc"][pick, 0], "sf": out["sf"][pick, 0]}
    arrays.update({"results_" + f: r[f] for f in r.dtype.names if f != "reserved"})
    arrays = {k: np.ascontiguousarray(v, np.float64) for k, v in arrays.items()}
    assert sum(v.nbytes for v in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    return sorted(arrays)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--batch", type=int, default=8192, help="streams (= frames per step) per GPU")
    ap.add_argument("--e2e-batch", type=int, default=0, help="streams per GPU in the host-buffer measurement (0 = the headline batch if the host has the memory)")
    ap.add_argument("--snr", type=float, default=20.0)
    ap.add_argument("--fft-mode", type=int, default=0)
    ap.add_argument("--distinct", type=int, default=8)
    ap.add_argument("--ref-frames", type=int, default=100)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-tail-split", action="store_true", help="A/B: do not cut the last frames of the OFDM launch into short CTAs")
    ap.add_argument("--cfo-hz", type=float, default=50.0, help="carrier offset of the secondary 'oscillator active' measurement (0 = skip); must keep the 5-frame ring periodic (multiples of 1/0.48 s)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0, a seeded sample of the streams) as DIR/<name>.npy, float64")
    a = ap.parse_args()
    if a.impl == "reference":
        reference_arm(a)
        return
    if a.warmup < 6:
        a.warmup = 6      # acquisition + 16-CIF de-interleaver fill + superframe sync must be over before the timed region

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    # ---- CPU baseline first (rank 0, N == 1), before CUDA is initialised in this process (the workers are forked)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        try:
            from oracle.bind import Ref
            if Ref.available():
                cores = max(1, int(effective_cores()["effective"]))
                n_procs = max(1, min(cores // 3, 48))
                log(f"cpu baseline: {n_procs} reference receivers x {a.ref_frames} frames")
                v, frames, busy, wall, ok, tot = run_reference_cpu(n_procs, a.ref_frames)
                cpu = {"value": v, "unit": "frames/s", "cores": cores, "kind": "reference", "cores_detail": effective_cores(),
                       "sample": f"{n_procs} concurrent unmodified reference RadioReceiver instances x {a.ref_frames} synthetic frames (same chain: FIC + one 96 kbit/s DAB+ sub-channel), KISS-FFT build, {busy:.1f} s",
                       "fib_crc_ok": ok, "fibs": tot}
                try:
                    cpu["stage_level"] = reference_stage_level()
                except Exception as e:  # noqa
                    cpu["stage_level"] = {"error": repr(e)}
                try:
                    cpu["stage_level_all_cores"] = reference_stage_level_all_cores(cores)
                except Exception as e:  # noqa
                    cpu["stage_level_all_cores"] = {"error": repr(e)}
                log(f"cpu baseline done: {v:.1f} frames/s")
        except Exception as e:  # noqa
            cpu = {"error": repr(e)}
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    numa_info = prefer_host_memory_near_gpu(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    pkg = load_pkg()
    S = a.batch
    # work descriptor: (first stream id of this rank) broadcast from rank 0 — the only collective on the path
    if world > 1:
        S = pkg.sharding.broadcast_descriptor([S], dev)[0]
    hbm_peak, peak_src, sm_max = measured_peaks()

    # ---- synthetic input: `distinct` periodic 5-frame rings, replicated to S stream buffers with per-stream AWGN
    rings = torch.from_numpy(make_rings(a.distinct).view(np.float32).reshape(a.distinct, RING_FRAMES * TF, 2)).to(dev)
    sig_pow = float((rings[:, 3000:190000] ** 2).sum(-1).mean())
    sigma = (sig_pow / (10 ** (a.snr / 10)) / 2) ** 0.5
    buf = torch.empty((S, BUF_LEN, 2), dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev); gen.manual_seed(0x5EED + rank)
    CH = 256
    for s0 in range(0, S, CH):
        n = min(CH, S - s0)
        idx = (torch.arange(s0, s0 + n, device=dev) + rank * S) % a.distinct
        blk = rings[idx] + torch.randn((n, RING_FRAMES * TF, 2), device=dev, generator=gen) * sigma
        buf[s0:s0 + n, :RING_FRAMES * TF] = blk
        buf[s0:s0 + n, RING_FRAMES * TF:] = blk[:, :BUF_LEN - RING_FRAMES * TF]
        del blk
    torch.cuda.synchronize()
    log(f"input ready: {S} streams x {BUF_LEN} samples")

    ctx = pkg.Context(n_streams=S, device=local, fft_mode=a.fft_mode, disable_coarse=True, n_subch_slots=1, max_subch_cu=SUBCH_CU, ofdm_tail_split=-1 if a.no_tail_split else 0)
    ctx.select_subchannel(0, SUBCH_CU, BITRATE, eep_profile_a=True, eep_level=3, dabplus=True)
    ext = torch.cuda.ExternalStream(ctx.cuda_stream(), device=dev)

    def buf_start_for(call):
        n = call + 1                      # call k decodes frame k+1 (frame 0 is consumed by the acquisition)
        return np.full(S, RING_FRAMES * TF * (n // RING_FRAMES), np.int64) if call > 0 else np.zeros(S, np.int64)

    call = 0
    for _ in range(a.warmup):
        ctx.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(call), BUF_LEN); call += 1
    ctx.sync()
    log("warm-up done")
    sampler = ClockSampler(local); sampler.start()
    sampler.ready.wait(20.0)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    l0 = ctx.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler.armed = True
    e0.record(ext)
    for _ in range(a.steps):
        ctx.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(call), BUF_LEN); call += 1
    ctx.join_lanes()       # the FIC / MSC / RS lane of the last steps runs on other streams: the closing event waits for it
    e1.record(ext)
    torch.cuda.synchronize()
    sampler.armed = False
    ms = e0.elapsed_time(e1)
    launches = ctx.kernel_launches() - l0
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    lt = torch.tensor([launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.barrier()
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
    sampler.stop_flag = True
    ms = float(t.item())
    value = world * S * a.steps / (ms * 1e-3)

    log(f"timed region done: {ms:.2f} ms for {a.steps} steps")
    # ---- validity of the timed work: one more step through the synchronous API, every stream must decode
    out = ctx.process(buf, BUF_LEN, buf_start_for(call), BUF_LEN, msc_stride=3 * BITRATE); call += 1
    r = out["results"]
    ok_frames = int((r["status"] == 0).sum()); fib_ok = int(sum(bin(int(m)).count("1") for m in r["fib_crc_mask"]))
    lf = int(r["n_logical"][:, 0].sum()); rs_unc = int((r["rs_uncorr_mask"][:, 0] != 0).sum()); rs_ev = int(r["n_rs_events"][:, 0].sum())
    check = {"frames_decoded": ok_frames, "streams": S, "fib_crc_ok": fib_ok, "fibs": 12 * S, "logical_frames": lf, "rs_attempts": rs_ev, "rs_uncorrectable_streams": rs_unc}
    if a.dump_outputs and rank == 0:
        names = dump_outputs(a.dump_outputs, a, pkg, local, S, buf, a.warmup + a.steps, buf_start_for)
        log(f"outputs of the last timed step written to {a.dump_outputs}: {', '.join(names)}")

    # ---- per-kernel device times over K more steady-state steps (CUDA events on the library's stream after every launch)
    ctx.profile(True)
    for _ in range(a.steps):
        ctx.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(call), BUF_LEN); call += 1
    ctx.sync()
    ctx.profile(False)
    prof = ctx.profile_read()
    clocks = sampler.summary()
    f_sm = (clocks["sm_mhz"] or sm_max) * 1e6
    kern = {k: {"ms_per_step": v["ms"] / a.steps, "launches_per_step": v["n"] / a.steps} for k, v in prof.items()}
    kms = prof["ofdm_demod_kernel"]["ms"] / prof["ofdm_demod_kernel"]["n"]
    ach = S * OFDM_BYTES_PER_FRAME / (kms * 1e-3) / 1e9
    traffic = None
    # DRAM bytes per frame of the kernel from the latest committed `ncu --set full` capture (profiles/rNN_ofdm_traffic.json)
    import glob
    tps = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ofdm_traffic.json")))
    tp = tps[-1] if tps else ""
    if tp:
        try:
            per = json.load(open(tp)).get("dram_bytes_per_frame")
            traffic = per * S if per else None
        except Exception:
            traffic = None
    roofline = {"kernel": "ofdm_demod_kernel", "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": traffic,
                "peak_source": peak_src, "bytes_per_launch": S * OFDM_BYTES_PER_FRAME, "ms_per_launch": kms,
                "frac_with_survey_bytes": S * SURVEY_BYTES_PER_FRAME / (kms * 1e-3) / 1e9 / hbm_peak,
                "share_of_step": kms / (sum(v["ms"] for v in prof.values()) / a.steps)}
    # Viterbi issue-slot figure (SURVEY §8d): 4 int-ops per ACS against 148 SM x 4 schedulers x 32 lanes x f_SM
    vms = sum(v_["ms"] for k_, v_ in prof.items() if k_.startswith("viterbi_kernel")) / a.steps
    acs_s = S * ACS_PER_FRAME / (vms * 1e-3)
    peak_ops = 148 * 4 * 32 * f_sm
    vit = {"kernel": "viterbi_kernel (FIC launch + MSC launch)", "bound": "issue", "achieved": acs_s * 4 / 1e12, "peak": peak_ops / 1e12, "unit": "Tint-op/s",
           "frac": acs_s * 4 / peak_ops, "acs_per_s": acs_s, "ms_per_step": vms, "f_sm_mhz": f_sm / 1e6,
           "note": "4 int-ops per add-compare-select (SURVEY 8d); the kernel packs two states per 32-bit lane-op"}

    # the same OFDM kernel in DABB_FFT_FMA arithmetic (contracted multiply-adds: <= 1e-6 relative on the spectra, softbits within
    # 1 LSB; integer outputs unchanged in the tests) timed alone through the stage-level entry point, for comparison
    fma = None
    try:
        Cc = pkg.dabb200.C
        ctx_f = pkg.Context(n_streams=1, device=local, fft_mode=pkg.FFT_FMA)
        softf = torch.empty((S, 75 * 3072), dtype=torch.int8, device=dev)
        prsf = torch.full((S,), TNULL + 305 + TF, dtype=torch.int64, device=dev)
        extf = torch.cuda.ExternalStream(ctx_f.cuda_stream(), device=dev)
        dur = []
        for i in range(5):
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            prsf.fill_(TNULL + 305 + TF * (1 + i % 4)); torch.cuda.synchronize()
            k0.record(extf)
            ctx_f._ck(ctx_f.lib.dabb_ofdm_demod(ctx_f.h, Cc.c_void_p(buf.data_ptr()), Cc.c_int64(BUF_LEN), Cc.c_void_p(prsf.data_ptr()), S, None, Cc.c_void_p(softf.data_ptr()), None, None))
            k1.record(extf); torch.cuda.synchronize()
            if i >= 2:
                dur.append(k0.elapsed_time(k1))
        fms = float(np.mean(dur))
        fma = {"ms_per_launch": fms, "achieved": S * OFDM_BYTES_PER_FRAME / (fms * 1e-3) / 1e9, "frac": S * OFDM_BYTES_PER_FRAME / (fms * 1e-3) / 1e9 / hbm_peak,
               "note": "ofdm_demod_kernel<FMA> alone (stage API, sync'd launches); the default and every other number in this line use the bit-exact arithmetic"}
        ctx_f.close(); del softf, prsf
    except Exception as e:  # noqa
        fma = {"error": repr(e)}
    roofline["fma_mode"] = fma
    log("kernel profile done")
    # ---- the other BASELINE.json configurations, as side measurements (the headline stays configs[3]/[4]) -------------------------------
    other = {}
    if world == 1 and not a.no_other_configs:
        # configs[1]: one stream, OFDM FFT + DQPSK kernel only (25 CTAs of 3 symbols each), device-resident frame
        try:
            Cc = pkg.dabb200.C
            c1 = pkg.Context(n_streams=1, device=local)
            soft1 = torch.empty((75 * 3072,), dtype=torch.int8, device=dev)
            prs1 = torch.full((1,), TNULL + 305 + TF, dtype=torch.int64, device=dev)
            x1 = torch.cuda.ExternalStream(c1.cuda_stream(), device=dev)
            dur = []
            for i in range(12):
                k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                k0.record(x1)
                c1._ck(c1.lib.dabb_ofdm_demod(c1.h, Cc.c_void_p(buf.data_ptr() + (i % 8) * BUF_LEN * 8), Cc.c_int64(BUF_LEN), Cc.c_void_p(prs1.data_ptr()), 1, None, Cc.c_void_p(soft1.data_ptr()), None, None))
                k1.record(x1); torch.cuda.synchronize()
                if i >= 4:
                    dur.append(k0.elapsed_time(k1))
            t1 = float(np.median(dur))
            other["configs[1] batch=1 OFDM kernel only"] = {"ms_per_frame": t1, "frames_per_s": 1e3 / t1, "hbm_gbs": OFDM_BYTES_PER_FRAME / (t1 * 1e-3) / 1e9,
                                                           "note": "one frame = 25 CTAs x (1 reference + 3 data symbols): latency-bound, 25 of 148 SMs busy; bit-exact vs the CPU in tests/test_gpu_stages.py"}
            c1.close(); del soft1, prs1
        except Exception as e:  # noqa
            other["configs[1] batch=1 OFDM kernel only"] = {"error": repr(e)}
        # configs[2]: batch 1024, full chain
        try:
            S2 = min(1024, S)
            c2 = pkg.Context(n_streams=S2, device=local, fft_mode=a.fft_mode, disable_coarse=True, n_subch_slots=1, max_subch_cu=SUBCH_CU)
            c2.select_subchannel(0, SUBCH_CU, BITRATE, eep_profile_a=True, eep_level=3, dabplus=True)
            x2 = torch.cuda.ExternalStream(c2.cuda_stream(), device=dev)
            cc = 0

            def bs2(call_):
                n_ = call_ + 1
                return np.full(S2, RING_FRAMES * TF * (n_ // RING_FRAMES), np.int64) if call_ > 0 else np.zeros(S2, np.int64)
            for _ in range(a.warmup):
                c2.process_async(buf.data_ptr(), BUF_LEN, bs2(cc), BUF_LEN); cc += 1
            c2.sync()
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record(x2)
            for _ in range(4 * a.steps):
                c2.process_async(buf.data_ptr(), BUF_LEN, bs2(cc), BUF_LEN); cc += 1
            c2.join_lanes(); k1.record(x2); torch.cuda.synchronize()
            ms2_ = k0.elapsed_time(k1) / (4 * a.steps)
            o2_ = c2.process(buf, BUF_LEN, bs2(cc), BUF_LEN, msc_stride=3 * BITRATE); cc += 1
            other["configs[2] batch=1024 full chain"] = {"ms_per_step": ms2_, "frames_per_s": S2 / (ms2_ * 1e-3),
                                                        "fic_crc_pass_rate": float(sum(bin(int(m)).count("1") for m in o2_["results"]["fib_crc_mask"])) / (12 * S2),
                                                        "frames_decoded": int((o2_["results"]["status"] == 0).sum())}
            c2.close()
        except Exception as e:  # noqa
            other["configs[2] batch=1024 full chain"] = {"error": repr(e)}
        # one stream through the host glue (RadioReceiver surface, n_streams = 1, all diagnostic taps on): what a welle-cli user gets
        try:
            import dabtx
            exe = os.path.join(ROOT, "welle.io_b200", "glue_test")
            if os.path.exists(exe):
                sig = dabtx.DabTx(seed=0x91).frames(120)
                fn = f"/tmp/bench_glue_{os.getpid()}.cf32"
                sig.tofile(fn)
                rr = subprocess.run([exe, fn, fn + ".out", "12"], capture_output=True, text=True, timeout=300)
                kv = dict(x.split("=") for x in rr.stdout.split())
                nfr = int(kv["fibs"]) // 12
                other["single stream through RadioReceiver glue"] = {"frames": nfr, "seconds": float(kv["seconds"]), "frames_per_s": nfr / float(kv["seconds"]), "fib_crc_ok": int(kv["ok"]),
                                                                     "note": "glue_test: memory-backed InputInterface -> RadioReceiver (host glue) -> dabb_process(n_streams = 1, CIR / constellation / null-symbol taps every frame); the reference's RadioReceiver does 137-205 frames/s on one stream (SURVEY 8d)"}
                for ext_ in ("", ".out.fibs", ".out.msc", ".out.rs"):
                    try:
                        os.remove(fn + ext_)
                    except OSError:
                        pass
        except Exception as e:  # noqa
            other["single stream through RadioReceiver glue"] = {"error": repr(e)}
        # acquisition of the whole batch at once (every stream runs the null search in the same call): the first dabb_process of a fresh context
        try:
            c3 = pkg.Context(n_streams=S, device=local, disable_coarse=True)
            x3 = torch.cuda.ExternalStream(c3.cuda_stream(), device=dev)
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record(x3); c3.process_async(buf.data_ptr(), BUF_LEN, np.zeros(S, np.int64), BUF_LEN); c3.join_lanes(); k1.record(x3); torch.cuda.synchronize()
            other["first call (acquisition of all streams)"] = {"ms": k0.elapsed_time(k1), "streams": S, "note": "sLevel warm-up + null search: one thread per stream, exact sequential arithmetic; once per stream"}
            c3.close()
        except Exception as e:  # noqa
            other["first call (acquisition of all streams)"] = {"error": repr(e)}
        log("other configurations done")

    # ---- e2e: host (pinned) IQ -> dabb_submit / dabb_collect (two steps in flight: H2D(n+1) | kernels(n) | D2H(n-1)) -> host results,
    # on the headline batch when the host has the memory for its pinned ring (BUF_LEN samples per stream), else the largest power-of-two
    # fraction that fits; cf32 (8 bytes per sample over PCIe) and the RAW u8 format of RTL-SDR recordings (2 bytes per sample)
    e2e = None
    if not a.no_e2e:
        def mem_available():
            """host bytes this process may still take: MemAvailable, further limited by the cgroup's memory limit (v2 or v1)"""
            avail = 64 << 30
            try:
                for ln in open("/proc/meminfo"):
                    if ln.startswith("MemAvailable"):
                        avail = int(ln.split()[1]) * 1024
            except Exception:
                pass
            for lim_f, cur_f in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                                 ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
                try:
                    lim = open(lim_f).read().strip()
                    if lim != "max" and int(lim) < (1 << 60):
                        avail = min(avail, int(lim) - int(open(cur_f).read().strip()))
                except Exception:
                    pass
            return max(avail, 0)
        Se = min(a.e2e_batch, S) if a.e2e_batch > 0 else S
        # pinned ring per rank: within the host's free memory (cgroup limit included), and never more than 80 GB over all ranks of the
        # box - the N = 1 run pins the headline batch (77.6 GB), N ranks share that (the pipelined path is PCIe-bound from a few hundred
        # frames per step on, and page-locking tens of GB on every rank at once takes minutes)
        budget = min(mem_available() * 0.45, 80e9) / max(1, min(world, 8))
        while Se > 64 and Se * BUF_LEN * 8 > budget:
            Se //= 2
        # PCIe host->device peak of this box: 1 GiB pinned -> device, best of 5
        pin = torch.empty(1 << 30, dtype=torch.uint8).pin_memory(); dst = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
        best = 0.0
        for _ in range(5):
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record(); dst.copy_(pin, non_blocking=True); p1.record(); torch.cuda.synchronize()
            best = max(best, (1 << 30) / (p0.elapsed_time(p1) * 1e-3) / 1e9)
        del pin, dst
        WIN = TF + 8192        # samples shipped per stream per step (one frame + sync margin)
        log(f"e2e: batch {Se} per GPU, pinned ring {Se * BUF_LEN * 8 / 1e9:.1f} GB (cf32), PCIe H2D peak {best:.1f} GB/s")

        def run_e2e(fmt_name):
            fmt = pkg.IQ_CF32 if fmt_name == "cf32" else pkg.IQ_U8
            bps = 8 if fmt_name == "cf32" else 2
            ctx_e = pkg.Context(n_streams=Se, device=local, fft_mode=a.fft_mode, disable_coarse=True, n_subch_slots=1, max_subch_cu=SUBCH_CU)
            ctx_e.select_subchannel(0, SUBCH_CU, BITRATE, eep_profile_a=True, eep_level=3, dabplus=True)
            if fmt_name == "cf32":
                host = torch.empty((Se, BUF_LEN, 2), dtype=torch.float32).pin_memory()
                for s0 in range(0, Se, 512):
                    host[s0:s0 + 512].copy_(buf[s0:s0 + 512])
            else:
                host = torch.empty((Se, BUF_LEN, 2), dtype=torch.uint8).pin_memory()
                for s0 in range(0, Se, 512):
                    host[s0:s0 + 512].copy_((buf[s0:s0 + 512] * 256.0 + 128.0).round().clamp(0, 255).to(torch.uint8))
            torch.cuda.synchronize()

            def args(c):
                n = c + 1
                if c == 0:
                    return host.data_ptr(), np.zeros(Se, np.int64), 3 * TF
                off = (n % RING_FRAMES) * TF
                return host.data_ptr() + off * bps, np.full(Se, n * TF, np.int64), min(WIN, BUF_LEN - off)

            def carry_of(c):
                # window c starts at (c + 1) TF; window c - 1 ended at its start + length: the overlap stays on the device (carry_samples)
                if c == 0:
                    return 0
                _, pbs, pbl = args(c - 1)
                return int(pbs[0] + pbl - (c + 1) * TF)
            ce = 0
            for _ in range(a.warmup):
                ptr, bs, bl = args(ce)
                ctx_e.process(ptr, BUF_LEN, bs, bl, iq_is_host=True, msc_stride=3 * BITRATE, sf_stride=15 * BITRATE, iq_format=fmt); ce += 1
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter(); h2d = 0; o = None; pipelined_started = False    # the warm-up used dabb_process: the first submit ships its whole window
            for k in range(a.steps):
                ptr, bs, bl = args(ce); cy = carry_of(ce) if pipelined_started else 0; ce += 1; h2d += Se * (bl - cy) * bps
                ctx_e.submit(ptr, BUF_LEN, bs, bl, msc_stride=3 * BITRATE, sf_stride=15 * BITRATE, iq_format=fmt, out=o if k >= 2 else None, carry=cy)   # result arrays recycled
                pipelined_started = True
                if k >= 1:
                    o = ctx_e.collect()
            o = ctx_e.collect()
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            te = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            dt = float(te.item())
            d2h = o["results"].nbytes + o["fibs"].nbytes + Se * 4 * 3 * BITRATE + Se * 15 * BITRATE
            res = {"value": world * Se * a.steps / dt, "unit": "frames/s", "h2d_bytes_per_step": h2d // a.steps, "d2h_bytes_per_step": d2h, "batch_frames_per_gpu": Se,
                   "frames_decoded_last_step": int((o["results"]["status"] == 0).sum()), "fib_crc_ok_last_step": int(sum(bin(int(m)).count("1") for m in o["results"]["fib_crc_mask"])),
                   "h2d_gbs_achieved_per_gpu": h2d / dt / 1e9, "h2d_frac_of_pcie_peak": h2d / dt / 1e9 / best if best else None}
            ctx_e.close(); del host
            return res
        try:
            e_cf = run_e2e("cf32")
            e2e = dict(e_cf)
            e2e["note"] = ("host pinned cf32 -> dabb_submit/dabb_collect, two steps in flight (H2D of step n+1 overlaps the kernels of step n and the result "
                           "read-back of step n-1; every sample crosses the link once: the 8192-sample window overlap is carried on the device); bound by the PCIe link: 1.57 MB of samples per frame")
            e2e["pcie_h2d_peak_gbs"] = best
            e2e["cf32_input"] = e_cf
        except Exception as e:  # noqa
            e2e = {"error": repr(e)}
        try:
            e2e["u8_input"] = run_e2e("u8")
            e2e["u8_input"]["note"] = "RAW u8 IQ (CRAWFile .u8.iq, the RTL-SDR format) shipped as bytes and converted on the device (SURVEY 8(f) rank 2): 0.39 MB per frame"
        except Exception as e:  # noqa
            e2e["u8_input"] = {"error": repr(e)}

    # ---- secondary measurement: the same streams with a carrier offset, so that the fine corrector is non-zero and every sample goes
    # through the oscillator table (the zero-offset streams of the headline run leave the oscillator at (1, 0), which the kernels skip)
    with_nco = None
    if a.cfo_hz and world == 1:
        try:
            ctx.close()
            ring_len = RING_FRAMES * TF
            nidx = torch.arange(BUF_LEN, device=dev, dtype=torch.float64) % ring_len
            ph = 2 * np.pi * a.cfo_hz * nidx / 2048000.0
            rc, rs = torch.cos(ph).to(torch.float32), torch.sin(ph).to(torch.float32)
            del nidx, ph
            for s0 in range(0, S, 64):
                blk = buf[s0:s0 + 64]
                re = blk[..., 0] * rc - blk[..., 1] * rs
                im = blk[..., 0] * rs + blk[..., 1] * rc
                blk[..., 0] = re; blk[..., 1] = im
                del re, im
            torch.cuda.synchronize()
            with_nco = {}
            for mode_name, mode in (("exact", pkg.NCO_EXACT), ("fast", pkg.NCO_FAST)):
                ctx2 = pkg.Context(n_streams=S, device=local, fft_mode=a.fft_mode, disable_coarse=True, n_subch_slots=1, max_subch_cu=SUBCH_CU, nco_mode=mode)
                ctx2.select_subchannel(0, SUBCH_CU, BITRATE, eep_profile_a=True, eep_level=3, dabplus=True)
                ext2 = torch.cuda.ExternalStream(ctx2.cuda_stream(), device=dev)
                c2 = 0
                for _ in range(a.warmup):
                    ctx2.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(c2), BUF_LEN); c2 += 1
                ctx2.sync()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record(ext2)
                for _ in range(a.steps):
                    ctx2.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(c2), BUF_LEN); c2 += 1
                ctx2.join_lanes()
                g1.record(ext2); torch.cuda.synchronize()
                ms2 = g0.elapsed_time(g1)
                ctx2.profile(True)
                for _ in range(a.steps):
                    ctx2.process_async(buf.data_ptr(), BUF_LEN, buf_start_for(c2), BUF_LEN); c2 += 1
                ctx2.sync(); ctx2.profile(False)
                pr2 = ctx2.profile_read()
                o2 = ctx2.process(buf, BUF_LEN, buf_start_for(c2), BUF_LEN, msc_stride=3 * BITRATE); c2 += 1
                r2 = o2["results"]
                k2 = pr2["ofdm_demod_kernel"]["ms"] / pr2["ofdm_demod_kernel"]["n"]
                with_nco[mode_name] = {"cfo_hz": a.cfo_hz, "nco_mode": mode_name, "value": S * a.steps / (ms2 * 1e-3), "unit": "frames/s", "ms_per_step": ms2 / a.steps, "ofdm_ms_per_launch": k2,
                            "ofdm_frac": S * OFDM_BYTES_PER_FRAME / (k2 * 1e-3) / 1e9 / hbm_peak,
                            "frames_decoded": int((r2["status"] == 0).sum()), "fib_crc_ok": int(sum(bin(int(m)).count("1") for m in r2["fib_crc_mask"])),
                            "fine_corr_median_hz": float(np.median(r2["fine_corr"])),
                            "oscillator_on_the_fly": int(ctx2.get_info(0)), "oscillator_table_mismatches": int(ctx2.get_info(1)),
                            "note": "same workload with a carrier offset: the numerically controlled oscillator (reference: 2 048 000-entry table lookup + complex multiply per sample; here evaluated on the fly after an exhaustive comparison with that table) is active for every stream"}
                ctx2.close()
        except Exception as e:  # noqa
            with_nco = {"error": repr(e)}
    roofline["oscillator_active"] = with_nco

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms / a.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+int16x2", "data": "synthetic",
                "config": dict(config_dict(a, None), host_numa=numa_info), "clocks": clocks, "e2e": e2e, "gpu_launches": int(lt.item()), "roofline": roofline, "roofline_viterbi": vit,
                "cpu_baseline": cpu, "check": check, "kernels": kern, "other_configs": other}
        print(json.dumps(line))
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
