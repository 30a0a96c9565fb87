#!/usr/bin/env python
"""bench.py -- throughput of the IQ sample-processing path on B200 (and the CPU reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...        (N > 1)

Workload (BASELINE.json configs[4], per-GPU share; configs[1] and [2] are its two halves):
every GPU holds `captures_per_gpu` independent synthetic 10 s captures (2.4 MS/s u8 I/Q,
48 MB each) resident in HBM and one "step" runs every capture through BOTH chains:
u8 -> Hann -> 1024-pt FFT -> |X|^2 -> mean (46 874 frames) and u8 -> /10 FIR -> discriminator ->
de-emphasis -> /5 FIR -> 48 kHz audio.  Captures are independent, so ranks share nothing on the
data path (weak scaling, no collective); torch.distributed only provides the barrier and the
max-over-ranks time.

`value` = complex samples entering the step per second, whole job, inputs resident in HBM.
`e2e`   = the same step through the C-ABI call that takes HOST buffers
          (b200sdr_batch_host: pinned host -> H2D -> kernels -> D2H of spectra and audio).
`roofline` = the dominant kernel (k_spectrum) alone: algorithmic 2 bytes per complex sample.
`cpu_baseline` / `--impl reference` = oracle/golden.c (fp32 build, kind "port": the reference
firmware has no DSP code of its own) on the host cores, same chains, bounded sample.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CAPTURE_BYTES = 48_000_000          # 10 s at 2.4 MS/s
CAPTURE_SAMPLES = CAPTURE_BYTES // 2
DUMP_BYTES = 60_000_000             # --dump-outputs: .npy payload of all files together (64 MB with headers and margin)
METRIC = "complex MS/s through u8->FFT-spectrum + u8->FIR->FM chains (batched 10 s captures)"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(directory, outputs, budget=DUMP_BYTES):
    """Write every (name, [rows, n] float32 tensor) of `outputs` to directory/<name>.npy.  An output that does not fit
    what is left of `budget` is cut to a fixed sample of its rows (np.random.default_rng(0), rows kept in order), so
    runs with the same arguments write the same rows.  Returns {name: rows written}."""
    import torch
    os.makedirs(directory, exist_ok=True)
    written = {}
    for name, t in outputs:
        rows, row_bytes = t.shape[0], t[0].numel() * 4
        keep = min(rows, budget // row_bytes)
        idx = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
        a = t.index_select(0, torch.from_numpy(idx).to(t.device)).cpu().numpy().astype(np.float32, copy=False)
        np.save(os.path.join(directory, name + ".npy"), a)
        budget -= keep * row_bytes
        written[name] = keep
    return written


def workload_config(B, world, fir_engine="tensor"):
    """The `config` object of BOTH arms (the GPU arm runs it whole; the CPU arm runs a bounded sample of it)."""
    return {"workload": "configs[4] per-GPU share (= configs[1] spectrum + configs[2] WBFM on every capture): "
                        f"{B} x 10 s captures (48 MB u8 I/Q each) per GPU, both chains per step",
            "captures_per_gpu": B, "capture_seconds": 10, "sample_rate": 2.4e6, "nfft": 1024, "hop": 512,
            "window": "hann", "fir_engine": fir_engine,
            "cache": f"inputs {B * CAPTURE_BYTES / 1e9:.1f} GB per GPU >> 126 MB L2 (no flush needed)",
            "parallelism": f"captures sharded over {world} GPU(s), no collective"}


def load_traffic_ratio():
    """DRAM bytes (read + write) per algorithmic byte of k_spectrum, from the newest tracked ncu capture
    (profiles/ncu_traffic.json, written by tools/ncu_summary.py --traffic): never a literal in this file."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        d = json.load(open(p))["k_spectrum"]
        return float(d["dram_bytes"]) / float(d["algorithmic_bytes"]), d.get("source", p)
    except (OSError, KeyError, ValueError, ZeroDivisionError):
        return None, None


# ------------------------------------------------------------------------------- CPU reference arm
class CpuArm:
    """oracle/golden.c (fp32 build) on the host cores, behind the word-granular ingest copy -- executed by the
    reference's OWN USB_ReadPacket (oracle/_ref, HAL_Driver/Src/stm32f7xx_ll_usb.c:792-803) when that build is
    present.  Checker / baseline only: nothing here is on the product path."""

    def __init__(self):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=True)
        import oracle_api
        self.api = oracle_api
        self.g = oracle_api.Golden(f32=True)
        self.copy_impl = "restated USB_ReadPacket (oracle/golden.c)"
        ref_so = os.path.join(ROOT, "oracle", "_ref", "libref_ingest.so")
        if os.path.exists(ref_so):
            ref = C.CDLL(ref_so)
            self.g.lib.gold_set_ingest_hook.argtypes = [C.c_void_p]
            self.g.lib.gold_set_ingest_hook(C.cast(ref.ref_copy_block, C.c_void_p))
            self._ref_keepalive = ref
            self.copy_impl = "the reference's own USB_ReadPacket (oracle/_ref)"
        self._captures = None

    def captures(self, distinct):
        """`distinct` synthetic 10 s captures (even: multitone, odd: FM -- the GPU arm's mix), made once."""
        if self._captures is None or self._captures[0] < distinct:
            parts = [self.g.synth(1, CAPTURE_BYTES, self.api.SYNTH_MULTITONE if c % 2 == 0 else self.api.SYNTH_WBFM, c)
                     for c in range(distinct)]
            self._captures = (distinct, np.concatenate(parts))
        return self._captures[1]

    def step(self, threads, captures_per_thread=1):
        """One bounded sample of the workload: threads x captures_per_thread 10 s captures, each through ingest copy +
        spectrum and ingest copy + WBFM.  Returns (samples, seconds of timed compute, spectrum s, wbfm s)."""
        n_blocks = threads * captures_per_thread
        distinct = min(n_blocks, 8)
        data = self.captures(distinct)
        ts = self.g.lib.gold_time_spectrum(data.ctypes.data, CAPTURE_SAMPLES, distinct, n_blocks, threads)
        tf = self.g.lib.gold_time_wbfm(data.ctypes.data, CAPTURE_SAMPLES, distinct, n_blocks, threads)
        return n_blocks * CAPTURE_SAMPLES, ts + tf, ts, tf

    def baseline(self, threads, target_seconds):
        samples, sec, ts, tf = self.step(threads, 1)
        reps = 1
        while sec < target_seconds * 0.5 and reps < 8:        # fast hosts: a second, larger sample
            reps *= 2
            samples, sec, ts, tf = self.step(threads, reps)
        return {"value": samples / sec / 1e6, "unit": "MS/s", "cores": threads, "kind": "port",
                "sample": f"{threads * reps} x 10 s captures (24 M samples each, the GPU arm's capture length) through ingest copy "
                          f"[{self.copy_impl}] + spectrum + WBFM [oracle/golden.c fp32 build], {threads} threads",
                "spectrum_MSps": samples / ts / 1e6, "wbfm_MSps": samples / tf / 1e6, "seconds": sec}

    def config0(self, threads_all):
        """BASELINE.md section 3 / configs[0]: ONE 262 144-byte block -> ingest copy -> cf32 -> Hann -> 1024-pt FFT ->
        |X|^2 -> mean of 255 frames; 1024 repetitions over 128 distinct buffers; 1 thread and all cores."""
        blk, distinct, reps = 262144, 128, 1024
        data = self.g.synth(distinct, blk, self.api.SYNTH_MULTITONE, 0)
        out = {"block_bytes": blk, "repetitions": reps, "distinct_buffers": distinct, "nproc": threads_all,
               "what": "configs[0]: one 256 KiB block -> ingest copy -> cf32 + 1024-pt Hann FFT power spectrum (255 frames), fp32 golden"}
        for label, th in (("1_thread", 1), ("all_cores", threads_all)):
            t = self.g.lib.gold_time_spectrum(data.ctypes.data, blk // 2, distinct, reps, th)
            out[label] = {"threads": th, "MSps": reps * (blk // 2) / t / 1e6, "us_per_block": t / reps * 1e6}
        return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    arm = CpuArm()
    arm.captures(min(threads, 8))                 # synthesis is not part of any timed step
    for _ in range(args.warmup):
        arm.step(threads, 1)
    samples = sec = ts = tf = 0.0
    for _ in range(args.steps):
        n, s_, a_, b_ = arm.step(threads, 1)
        samples += n; sec += s_; ts += a_; tf += b_
    v = samples / sec / 1e6
    res = {"value": v, "unit": "MS/s", "cores": threads, "kind": "port",
           "sample": f"each step = {threads} x 10 s captures (24 M samples each) through ingest copy [{arm.copy_impl}] + spectrum + "
                     f"WBFM [oracle/golden.c fp32 build], {threads} threads; {args.steps} steps",
           "spectrum_MSps": samples / ts / 1e6, "wbfm_MSps": samples / tf / 1e6, "seconds": sec,
           "config0": arm.config0(threads)}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * sec / max(args.steps, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.captures_per_gpu, world, args.fir_engine),
            "cpu_baseline": res, "e2e": {"value": v, "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bind_to_gpu_numa_node(gpu_index):
    """Run this rank (and first-touch its pinned buffers) on the NUMA node the GPU hangs off, so
    the host->device copies of several ranks do not cross the socket interconnect."""
    try:
        multi_node = "-" in open("/sys/devices/system/node/online").read() or "," in open("/sys/devices/system/node/online").read()
    except OSError:
        multi_node = False
    if os.environ.get("B200_BENCH_NUMA", "1" if multi_node else "0") != "1":
        return
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(gpu_index)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        bdf = out[-12:] if len(out) >= 12 else out          # 00000000:1B:00.0 -> 0000:1b:00.0
        cpus = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
    except Exception:
        pass


# ---------------------------------------------------------------------------------------- GPU arm
def split_capture_probe(pkg, sharding, sdr, dist, torch, rank, world):
    """One 10 s capture split in time over the ranks (SURVEY 8e): every rank runs k_spectrum over its own
    frames and ONE kernel reduces the partial sums, pushes them to every peer over NVLink peer memory and
    adds the ranks' contributions in rank order.  Returns a small dict for the JSON line.  Every rank
    makes the same sequence of collective calls whatever fails locally (failures are agreed on with an
    all-reduce), so a problem here can never desynchronise the rest of the benchmark."""
    def all_ok(ok):
        f = torch.tensor([1 if ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(f, op=dist.ReduceOp.MIN)
        return bool(f.item())

    err, handle = "", None
    try:
        handle = sdr.exchange_create(world, rank)
    except Exception as e:
        err = str(e)
    handles = [None] * world
    dist.all_gather_object(handles, handle)                                  # plumbing: 64-byte IPC handles
    try:
        if any(h is None for h in handles):
            raise RuntimeError(err or "a peer could not create its mailbox")
        sdr.exchange_connect(handles)
        cap = torch.empty(CAPTURE_BYTES, dtype=torch.uint8, device="cuda")
        out = torch.zeros(1024, dtype=torch.float32, device="cuda")
        whole = torch.empty(1024, dtype=torch.float32, device="cuda")
        sdr.synth_fill_dev(cap.data_ptr(), 1, CAPTURE_BYTES, pkg.SYNTH_MULTITONE, first_capture=999)  # same capture everywhere
        sdr.batch_spectrum_dev(cap.data_ptr(), 1, CAPTURE_BYTES, whole.data_ptr())                   # single-GPU answer
        sdr.sync()
        ok = True
    except Exception as e:
        err, ok = str(e), False
    if not all_ok(ok):
        return {"error": ("setup: " + err)[:300]}
    frames = (CAPTURE_SAMPLES - 1024) // 512 + 1
    b0, b1, _, _ = sharding.split_capture_bytes(CAPTURE_BYTES, rank, world)
    iters, dt = 20, 0.0
    try:
        for i in range(3 + iters):
            if i == 3:
                torch.cuda.synchronize()
                t0 = time.perf_counter()
            sdr.split_spectrum_dev(cap.data_ptr() + b0, b1 - b0, frames, out.data_ptr())
            sdr.exchange_wait()                                              # bounded: FAIL after ~5 s, never a hang
        dt = (time.perf_counter() - t0) / iters
    except Exception as e:
        err, ok = str(e), False
    if not all_ok(ok):
        return {"error": ("exchange: " + err)[:300]}
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    gathered = [torch.zeros_like(out) for _ in range(world)]
    dist.all_gather(gathered, out)
    same = all(torch.equal(gathered[0], g) for g in gathered)
    rel = float(((out - whole).abs() / whole).max())
    try:
        sdr.exchange_destroy()
    except Exception:
        pass
    return {"what": "one 10 s capture split over the ranks: k_spectrum on each slice + ONE fused finalize / NVLink "
                    "peer-memory all-reduce kernel (no library collective)",
            "us_per_capture": float(t.item()) * 1e6, "MSps": CAPTURE_SAMPLES / float(t.item()) / 1e6,
            "bitwise_identical_on_all_ranks": bool(same), "max_rel_diff_vs_single_gpu_spectrum": rel}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every timed section")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--captures-per-gpu", type=int, default=512)
    ap.add_argument("--e2e-captures", type=int, default=64)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--parity-captures", type=int, default=64, help="captures per rank recomputed one at a time (bitwise check)")
    ap.add_argument("--config4-waves", type=int, default=8, help="N=1 only: waves of captures-per-gpu captures (8 x 512 = configs[4]); 0 = skip")
    ap.add_argument("--fir-engine", default="tensor", choices=["tensor", "fp32"],
                    help="stage-1 FIR engine of the batched WBFM chain the step (and e2e) runs: tensor = exact u8 x s8 tcgen05 product "
                         "(csrc/wbfm_tc.cuh), fp32 = CUDA-core scatter FIR (csrc/wbfm.cuh); the other engine is timed beside it")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned on rank 0 (its captures are the job's first "
                         "captures-per-gpu) as DIR/spectrum.npy [captures, 1024] and DIR/wbfm_audio.npy [captures, 48 kHz "
                         "samples], float32; outputs over the %d-byte budget are a fixed seeded sample of their captures" % DUMP_BYTES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    bind_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    importlib.import_module("stm32f7-rtlsdr_b200.build").build()
    pkg = importlib.import_module("stm32f7-rtlsdr_b200")
    sharding = importlib.import_module("stm32f7-rtlsdr_b200.sharding")
    engines = {"tensor": pkg.FIR_ENGINE_TENSOR, "fp32": pkg.FIR_ENGINE_FP32}
    other_engine = "fp32" if args.fir_engine == "tensor" else "tensor"
    sdr = pkg.B200Sdr(device=local_rank, chains=pkg.CHAIN_SPECTRUM | pkg.CHAIN_WBFM, fir_engine=engines[args.fir_engine])
    sdr_other = pkg.B200Sdr(device=local_rank, chains=pkg.CHAIN_WBFM, fir_engine=engines[other_engine])  # timed beside it

    B = args.captures_per_gpu
    lo, hi = sharding.shard_range(B * world, rank, world)   # this rank's captures of the whole job
    assert hi - lo == B
    # torch owns the big device buffers (plumbing); the library only sees raw pointers
    iq = torch.empty(B * CAPTURE_BYTES, dtype=torch.uint8, device="cuda")
    spec = torch.empty(B * 1024, dtype=torch.float32, device="cuda")
    n_audio = pkg.wbfm_audio_len(CAPTURE_BYTES)
    audio = torch.empty(B * n_audio, dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    for c0 in range(0, B, 64):                               # even captures multitone, odd FM
        n = min(64, B - c0)
        for c in range(c0, c0 + n):
            kind = pkg.SYNTH_MULTITONE if (lo + c) % 2 == 0 else pkg.SYNTH_WBFM
            sdr.synth_fill_dev(iq.data_ptr() + c * CAPTURE_BYTES, 1, CAPTURE_BYTES, kind, first_capture=lo + c)
    sdr.sync()

    n_am = pkg.am_audio_len(CAPTURE_BYTES)
    am_audio = torch.empty(B * n_am, dtype=torch.float32, device="cuda")

    def step(which=3):
        if which & 1:
            sdr.batch_spectrum_dev(iq.data_ptr(), B, CAPTURE_BYTES, spec.data_ptr())
        if which & 2:
            sdr.batch_wbfm_dev(iq.data_ptr(), B, CAPTURE_BYTES, audio.data_ptr())
        if which & 4:   # secondary chain (config[3]); not part of the headline step
            sdr.batch_am_dev(iq.data_ptr(), B, CAPTURE_BYTES, am_audio.data_ptr())

    def timed(which, steps):
        barrier()
        sdr.timer_start()
        for _ in range(steps):
            step(which)
        ms = sdr.timer_stop_ms()        # CUDA events on the library's compute stream
        barrier()
        return max_over_ranks(ms)

    sampler = ClockSampler(local_rank)   # polls nvidia-smi while the device-timed regions run (incl. warm-up:
    sampler.start()                      # same load); stopped before e2e, whose PCIe copies the polling perturbs
    for _ in range(args.warmup):
        step()
    sdr.sync()
    l0 = sdr.kernel_launches()
    ms_total = timed(3, args.steps)
    launches = sdr.kernel_launches() - l0
    if args.dump_outputs and rank == 0:   # spec / audio hold the last timed step's results until the next step runs
        dumped = dump_outputs(args.dump_outputs, [("spectrum", spec.view(B, 1024)), ("wbfm_audio", audio.view(B, n_audio))])
        sys.stderr.write(f"dump-outputs: captures written {dumped} to {args.dump_outputs}\n")
    ms_spec = timed(1, args.steps)
    ms_fm = timed(2, args.steps)
    # the same WBFM batch through the OTHER stage-1 FIR engine (own context, own stream), and how far its audio is from
    # the step's engine (both are within the parity tolerance of the float64 golden model; tests/test_gpu_parity.py)
    audio_other = torch.empty(B * n_audio, dtype=torch.float32, device="cuda")
    for _ in range(2):
        sdr_other.batch_wbfm_dev(iq.data_ptr(), B, CAPTURE_BYTES, audio_other.data_ptr())
    sdr_other.sync()
    barrier()
    sdr_other.timer_start()
    for _ in range(args.steps):
        sdr_other.batch_wbfm_dev(iq.data_ptr(), B, CAPTURE_BYTES, audio_other.data_ptr())
    ms_fm_other = max_over_ranks(sdr_other.timer_stop_ms())
    sdr_other.sync()
    n_cmp = min(B, 64) * n_audio
    engines_max_diff = float((audio_other[:n_cmp] - audio[:n_cmp]).abs().max())
    sys.stderr.write(f"engines: max |audio| {float(audio[:n_cmp].abs().max()):.6f} / {float(audio_other[:n_cmp].abs().max()):.6f}, "
                     f"max difference {engines_max_diff:.3e}\n")
    del audio_other
    clocks = sampler.stop()
    step(4)
    sdr.sync()
    ms_am = timed(4, args.steps)

    # K2 alone (u8 -> cf32, 2 B in + 8 B out per sample): the one HBM-bound kernel of the path, as a
    # reference for what the memory system gives this access pattern
    Bc = min(B, 48)
    cf = torch.empty(Bc * CAPTURE_BYTES, dtype=torch.float32, device="cuda")
    conv = sdr.lib.b200sdr_convert_cf32_dev
    for _ in range(2):
        conv(sdr.ctx, iq.data_ptr(), Bc * CAPTURE_BYTES, 0, cf.data_ptr())
    barrier()
    sdr.timer_start()
    for _ in range(args.steps):
        conv(sdr.ctx, iq.data_ptr(), Bc * CAPTURE_BYTES, 0, cf.data_ptr())
    ms_conv = max_over_ranks(sdr.timer_stop_ms())
    conv_gbs = 10.0 * Bc * CAPTURE_SAMPLES * args.steps / (ms_conv * 1e-3) / 1e9
    del cf

    # K0 alone (test-mode counter check: 1 byte read per byte, nothing written), on counter captures -- what the
    # firmware's stream really carries (RTLSDR_set_test_mode(phost, 1), usbh_rtlsdr.c:901).  The call includes its
    # own result read-back (16 bytes per capture) and stream synchronisation.
    Bk = min(B, 128)
    ms_cnt, cnt_breaks = float("nan"), -1
    try:  # informative chain: whatever goes wrong here must not cost the headline line
        cnt = torch.empty(Bk * CAPTURE_BYTES, dtype=torch.uint8, device="cuda")
        for c in range(Bk):
            sdr.synth_fill_dev(cnt.data_ptr() + c * CAPTURE_BYTES, 1, CAPTURE_BYTES, pkg.SYNTH_COUNTER, first_capture=c)
        for _ in range(2):
            n_breaks, _first = sdr.counter_check_dev(cnt.data_ptr(), Bk, CAPTURE_BYTES)
        sdr.timer_start()                      # no barrier in here: a rank that failed above must not strand the others
        for _ in range(args.steps):
            n_breaks, _first = sdr.counter_check_dev(cnt.data_ptr(), Bk, CAPTURE_BYTES)
        ms_cnt = sdr.timer_stop_ms()
        cnt_breaks = int(n_breaks.sum())
        del cnt
    except Exception as exc:  # noqa: BLE001
        sys.stderr.write(f"counter-check chain skipped: {exc}\n")
    ms_cnt = max_over_ranks(ms_cnt if ms_cnt == ms_cnt else 0.0)   # every rank takes part in the reduction
    cnt_gbs = 2.0 * Bk * CAPTURE_SAMPLES * args.steps / (ms_cnt * 1e-3) / 1e9 if ms_cnt > 0 else 0.0

    samples_step = B * CAPTURE_SAMPLES * world              # whole job, per step
    value = samples_step * args.steps / (ms_total * 1e-3) / 1e6
    hbm_peak, peak_src = load_peaks()
    spec_gbs = 2.0 * B * CAPTURE_SAMPLES * args.steps / (ms_spec * 1e-3) / 1e9            # per GPU
    fm_bytes = 2.0 + 4.0 * 48000.0 / 2400000.0
    fm_gbs = fm_bytes * B * CAPTURE_SAMPLES * args.steps / (ms_fm * 1e-3) / 1e9
    fm_other_gbs = fm_bytes * B * CAPTURE_SAMPLES * args.steps / (ms_fm_other * 1e-3) / 1e9
    am_bytes = 2.0 + 4.0 * 8000.0 / 2400000.0
    am_gbs = am_bytes * B * CAPTURE_SAMPLES * args.steps / (ms_am * 1e-3) / 1e9

    # ---- parity of the sharded batch (SURVEY 4(iv)): every capture of this rank's shard recomputed ONE AT A TIME must
    # give bitwise the spectrum / audio it got inside the batch of B (the summation tree follows from the capture
    # length only, csrc/plan.h), and a capture computed on every GPU must give the same bits on every GPU.
    step(3)
    sdr.sync()
    one_spec = torch.empty(1024, dtype=torch.float32, device="cuda")
    one_audio = torch.empty(n_audio, dtype=torch.float32, device="cuda")
    spec2, audio2 = spec.view(B, 1024), audio.view(B, n_audio)
    n_checked, n_equal = 0, 0
    for c in range(0, B, max(1, B // max(1, args.parity_captures))):
        sdr.batch_spectrum_dev(iq.data_ptr() + c * CAPTURE_BYTES, 1, CAPTURE_BYTES, one_spec.data_ptr())
        sdr.batch_wbfm_dev(iq.data_ptr() + c * CAPTURE_BYTES, 1, CAPTURE_BYTES, one_audio.data_ptr())
        sdr.sync()
        n_checked += 1
        n_equal += int(torch.equal(one_spec, spec2[c]) and torch.equal(one_audio, audio2[c]))
    # the job's capture 0 and 1 (multitone, FM) recomputed on EVERY rank: digests must agree across GPUs and across N
    probe = torch.empty(2 * CAPTURE_BYTES, dtype=torch.uint8, device="cuda")
    sdr.synth_fill_dev(probe.data_ptr(), 1, CAPTURE_BYTES, pkg.SYNTH_MULTITONE, first_capture=0)
    sdr.synth_fill_dev(probe.data_ptr() + CAPTURE_BYTES, 1, CAPTURE_BYTES, pkg.SYNTH_WBFM, first_capture=1)
    p_spec = torch.empty(2 * 1024, dtype=torch.float32, device="cuda")
    p_audio = torch.empty(2 * n_audio, dtype=torch.float32, device="cuda")
    sdr.batch_spectrum_dev(probe.data_ptr(), 2, CAPTURE_BYTES, p_spec.data_ptr())
    sdr.batch_wbfm_dev(probe.data_ptr(), 2, CAPTURE_BYTES, p_audio.data_ptr())
    sdr.sync()
    import hashlib
    digest = hashlib.sha256(p_spec.cpu().numpy().tobytes() + p_audio.cpu().numpy().tobytes()).hexdigest()[:16]
    del probe
    counts = torch.tensor([n_checked, n_equal], dtype=torch.int64, device="cuda")
    digests = [digest]
    if world > 1:
        dist.all_reduce(counts)
        digests = [None] * world
        dist.all_gather_object(digests, digest)
    if rank == 0 and B >= 2:   # rank 0 owns the job's captures 0 and 1: the probe must equal what the batch gave them
        in_batch = hashlib.sha256(spec2[:2].cpu().numpy().tobytes() + audio2[:2].cpu().numpy().tobytes()).hexdigest()[:16]
    else:
        in_batch = None
    parity = {"bitwise": bool(int(counts[0]) == int(counts[1]) and len(set(digests)) == 1 and in_batch in (None, digest)),
              "captures_recomputed_alone": int(counts[0]), "equal_to_batch_result": int(counts[1]),
              "probe_digest_per_rank": digests, "probe_digest_in_rank0_batch": in_batch,
              "what": "spectrum + WBFM audio of captures recomputed one at a time == their results inside the batch of "
                      f"{B}; captures 0/1 of the job recomputed on every rank: sha256 equal on all GPUs (and across runs at other N)"}

    # ---- configs[4] literally on ONE GPU: 4096 captures = 8 waves of 512, each wave's captures regenerated on the device
    # (196.6 GB does not fit one B200); chains timed per wave with CUDA events, generation not timed ------------------
    config4 = None
    if world == 1 and args.config4_waves > 0:
        ms_waves, t_wall = 0.0, time.perf_counter()
        for w in range(args.config4_waves):
            if w > 0:      # wave 0 is what is resident already (captures 0..B-1 of the job)
                for c in range(B):
                    kind = pkg.SYNTH_MULTITONE if (w * B + c) % 2 == 0 else pkg.SYNTH_WBFM
                    sdr.synth_fill_dev(iq.data_ptr() + c * CAPTURE_BYTES, 1, CAPTURE_BYTES, kind, first_capture=w * B + c)
                sdr.sync()
            sdr.timer_start()
            step(3)
            ms_waves += sdr.timer_stop_ms()
        n_cap4 = args.config4_waves * B
        config4 = {"captures": n_cap4, "waves": args.config4_waves, "captures_per_wave": B, "ms_chains": ms_waves,
                   "MSps": n_cap4 * CAPTURE_SAMPLES / (ms_waves * 1e-3) / 1e6,
                   "wall_s_with_regeneration": time.perf_counter() - t_wall,
                   "last_wave_checksum": float(spec2[B - 1].sum()),
                   "note": "configs[4] on one GPU: waves share one 24.6 GB input buffer, regenerated between waves (not timed)"}

    # ---- N > 1 only, informative: the one exchange step the path can have -- ONE 10 s capture split in time
    # across the ranks, bin sums combined by the fused finalize + NVLink peer-memory all-reduce kernel
    # (csrc/exchange.cuh).  Not part of `value`; a failure here is reported, never fatal. --------------------
    split = None
    if world > 1:
        split = split_capture_probe(pkg, sharding, sdr, dist, torch, rank, world)

    # ---- end to end through the host-buffer entry point --------------------------------------
    E = min(args.e2e_captures, B)
    hp, h_iq = sdr.pinned_alloc(E * CAPTURE_BYTES)
    sp, h_spec = sdr.pinned_alloc(E * 1024 * 4, np.float32)
    fp, h_fm = sdr.pinned_alloc(E * n_audio * 4, np.float32)
    sdr.lib.b200sdr_copy_to_host(sdr.ctx, h_iq.ctypes.data, iq.data_ptr(), E * CAPTURE_BYTES)
    for _ in range(2):
        sdr.batch_host(pkg.CHAIN_SPECTRUM | pkg.CHAIN_WBFM, h_iq, E, CAPTURE_BYTES, spectrum=h_spec, wbfm=h_fm)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        sdr.batch_host(pkg.CHAIN_SPECTRUM | pkg.CHAIN_WBFM, h_iq, E, CAPTURE_BYTES, spectrum=h_spec, wbfm=h_fm)
    torch.cuda.synchronize()
    e2e_mine = time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_mine)
    e2e_value = E * CAPTURE_SAMPLES * world * e2e_steps / e2e_s / 1e6
    checksum = float(h_spec[:1024].sum()) + float(h_fm[:1000].sum())

    # what the host can feed: every rank at once does a PLAIN pinned cudaMemcpyAsync H2D of the same bytes from the same
    # buffer (no kernels, no D2H) -- the ceiling b200sdr_batch_host is judged against (PCIe switch / root-complex topology
    # and host memory are shared by the ranks, so the aggregate is not N x the single-GPU figure)
    dst = torch.empty(E * CAPTURE_BYTES, dtype=torch.uint8, device="cuda")
    src_t = torch.from_numpy(h_iq)          # the library's pinned buffer: cudaMemcpyAsync treats it as pinned
    for _ in range(2):
        dst.copy_(src_t, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        dst.copy_(src_t, non_blocking=True)
    torch.cuda.synchronize()
    h2d_mine = time.perf_counter() - t0
    h2d_s = max_over_ranks(h2d_mine)
    del dst
    per_rank = [(E * CAPTURE_BYTES * e2e_steps / e2e_mine / 1e9, E * CAPTURE_BYTES * e2e_steps / h2d_mine / 1e9)]
    if world > 1:
        per_rank = [None] * world
        dist.all_gather_object(per_rank, (E * CAPTURE_BYTES * e2e_steps / e2e_mine / 1e9, E * CAPTURE_BYTES * e2e_steps / h2d_mine / 1e9))
    h2d_agg = E * CAPTURE_BYTES * world * e2e_steps / h2d_s / 1e9
    e2e_agg = E * CAPTURE_BYTES * world * e2e_steps / e2e_s / 1e9
    for p in (hp, sp, fp):
        sdr.pinned_free(p)

    # ---- streaming ingest through process_samples (ring -> H2D -> chains), labelled separately:
    # launch- and PCIe-bound, what a live 2.4 MS/s dongle would exercise (needs 4.8 MB/s) ------
    ingest = None
    if rank == 0:
        blk = 262144
        s2 = pkg.B200Sdr(device=local_rank, chains=pkg.CHAIN_SPECTRUM | pkg.CHAIN_WBFM, slot_bytes=blk, ring_slots=8,
                         audio_capacity=1 << 22)
        src = pkg.synth_fill_host(1, blk * 16, pkg.SYNTH_WBFM, 0)
        n_blocks, busy = 512, 0
        for i in range(32):
            while s2.process_samples(src[(i % 16) * blk:(i % 16 + 1) * blk], allow_busy=True) == pkg.BUSY:
                pass
        s2.sync()
        s2.get_audio(pkg.CHAIN_WBFM, 1 << 22)
        t0 = time.perf_counter()
        for i in range(n_blocks):
            view = src[(i % 16) * blk:(i % 16 + 1) * blk]
            while s2.process_samples(view, allow_busy=True) == pkg.BUSY:
                busy += 1  # every ring slot in flight: poll again (the audio FIFO holds the whole run)
        s2.sync()
        dt = time.perf_counter() - t0
        ingest = {"api": "process_samples", "block_bytes": blk, "blocks": n_blocks, "MSps": n_blocks * blk / 2 / dt / 1e6,
                  "us_per_block": dt / n_blocks * 1e6, "busy_returns": busy, "realtime_factor_at_2.4MSps": n_blocks * blk / 2 / dt / 2.4e6}
        s2.close()
        # the firmware's own cadence from a plain C caller (examples/firmware_cadence.c): ONE 512-byte
        # buffer re-armed after every process_samples() call, spectrum read back every 4096 blocks
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", str(local_rank)))
        # the same from a plain C caller (examples/ingest_bench.c), 256 KiB slots: process_samples (the block is copied into
        # the pinned slot) and ring_acquire / ring_commit (zero-copy: the producer fills the slot, only the enqueue is timed)
        ib = os.path.join(ROOT, "build", "ingest_bench")
        if os.path.exists(ib):
            try:
                out = subprocess.run([ib, str(blk), "2048"], capture_output=True, text=True, timeout=120, env=env).stdout
                for ln in out.splitlines():
                    if ln.startswith("INGEST"):
                        kv = dict(t.split("=") for t in ln.split()[1:])
                        ingest["c_caller_" + kv["mode"]] = {"us_per_block": float(kv["us_per_block"]), "GBps": float(kv["GBps"]),
                                                            "MSps": float(kv["MSps"]), "busy_returns": int(kv["busy"]),
                                                            "realtime_factor_at_2.4MSps": float(kv["realtime"])}
            except Exception as e:  # the probe is informative only
                ingest["c_caller"] = {"error": str(e)[:200]}
        fw = os.path.join(ROOT, "build", "firmware_cadence")
        if os.path.exists(fw):
            for key, argv in (("firmware_512B_coalesced", ["96000000", "512", "0", "262144", "4096"]),
                              ("firmware_512B_per_block", ["2048000", "512", "4", "262144", "4096"])):
                try:
                    out = subprocess.run([fw] + argv, capture_output=True, text=True, timeout=120, env=env).stdout
                    kv = dict(t.split("=") for t in out.split() if "=" in t)
                    ingest[key] = {"MSps": float(kv["MSps"]), "us_per_block": float(kv["us_per_block"]),
                                   "realtime_factor_at_2.4MSps": float(kv["realtime"]), "blocks": int(kv["blocks"])}
                except Exception as e:  # the probe is informative only
                    ingest[key] = {"error": str(e)[:200]}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        arm = CpuArm()
        cpu = arm.baseline(os.cpu_count() or 1, 12.0)
        cpu["config0"] = arm.config0(os.cpu_count() or 1)

    traffic_ratio, traffic_src = load_traffic_ratio()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "MS/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(B, world, args.fir_engine),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "MS/s", "h2d_bytes_per_step": E * CAPTURE_BYTES,
                    "d2h_bytes_per_step": E * (1024 + n_audio) * 4, "captures_per_step": E, "steps": e2e_steps,
                    "api": "b200sdr_batch_host (pinned host -> H2D -> kernels -> D2H)", "checksum": checksum,
                    "h2d_GBps_aggregate": e2e_agg, "h2d_GBps_per_rank": [round(a, 2) for a, _ in per_rank],
                    "h2d_ceiling": {"what": "all ranks at once: plain pinned cudaMemcpyAsync H2D of the same bytes, no kernels",
                                    "GBps_aggregate": h2d_agg, "GBps_per_rank": [round(b, 2) for _, b in per_rank]},
                    "frac_of_h2d_ceiling": e2e_agg / h2d_agg},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": "k_spectrum (+k_spectrum_finalize)", "achieved": spec_gbs, "peak": hbm_peak,
                         "unit": "GB/s", "frac": spec_gbs / hbm_peak,
                         "traffic": (traffic_ratio * 2.0 * B * CAPTURE_SAMPLES) if traffic_ratio else None,  # bytes per launch
                         "traffic_source": traffic_src,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_sample": 2.0,
                         "note": "FP32-pipe bound, not HBM bound (DESIGN.md 5.1): 1028 FP32-pipe cycles per 1024-pt frame per SM "
                                 "sub-partition for 512 new samples",
                         "fp32_ceiling_GBps": 2.0 * 148 * 4 * (clocks.get("sm_mhz") or 1965.0) * 1e6 * 512 / 1028 / 1e9,
                         "frac_of_fp32_ceiling": spec_gbs / (2.0 * 148 * 4 * (clocks.get("sm_mhz") or 1965.0) * 1e6 * 512 / 1028 / 1e9)},
            "chains": {
                "spectrum": {"ms_per_step": ms_spec / args.steps, "MSps_per_gpu": B * CAPTURE_SAMPLES * args.steps / (ms_spec * 1e-3) / 1e6,
                             "GBps": spec_gbs, "hbm_frac": spec_gbs / hbm_peak, "hbm_frac_nominal_8TBps": spec_gbs / 8000.0},
                "wbfm": {"ms_per_step": ms_fm / args.steps, "MSps_per_gpu": B * CAPTURE_SAMPLES * args.steps / (ms_fm * 1e-3) / 1e6,
                         "GBps": fm_gbs, "hbm_frac": fm_gbs / hbm_peak, "hbm_frac_nominal_8TBps": fm_gbs / 8000.0,
                         "algorithmic_bytes_per_sample": fm_bytes, "fir_engine": args.fir_engine,
                         "kernel": "k_wbfm_tc" if args.fir_engine == "tensor" else "k_wbfm"},
                "wbfm_" + other_engine + "_engine": {
                    "ms_per_step": ms_fm_other / args.steps, "MSps_per_gpu": B * CAPTURE_SAMPLES * args.steps / (ms_fm_other * 1e-3) / 1e6,
                    "GBps": fm_other_gbs, "hbm_frac": fm_other_gbs / hbm_peak, "hbm_frac_nominal_8TBps": fm_other_gbs / 8000.0,
                    "algorithmic_bytes_per_sample": fm_bytes, "kernel": "k_wbfm_tc" if other_engine == "tensor" else "k_wbfm",
                    "max_abs_audio_difference_between_engines": engines_max_diff,
                    "note": "the same batch through the other stage-1 FIR engine (cfg.fir_engine); not part of `value`"},
                "convert_cf32": {"ms_per_step": ms_conv / args.steps, "MSps_per_gpu": Bc * CAPTURE_SAMPLES * args.steps / (ms_conv * 1e-3) / 1e6,
                                 "GBps": conv_gbs, "hbm_frac": conv_gbs / hbm_peak, "algorithmic_bytes_per_sample": 10.0,
                                 "note": "K2 alone over %d captures: HBM-bound reference, not part of `value`" % Bc},
                "counter_check": {"ms_per_step": ms_cnt / args.steps, "MSps_per_gpu": cnt_gbs * 1e3 / 2.0,
                                  "GBps": cnt_gbs, "hbm_frac": cnt_gbs / hbm_peak, "hbm_frac_nominal_8TBps": cnt_gbs / 8000.0,
                                  "algorithmic_bytes_per_sample": 2.0, "breaks_found": cnt_breaks,
                                  "note": "K0 alone over %d counter captures (the firmware's test-mode stream): HBM-bound, "
                                          "not part of `value`" % Bk},
                "am": {"ms_per_step": ms_am / args.steps, "MSps_per_gpu": B * CAPTURE_SAMPLES * args.steps / (ms_am * 1e-3) / 1e6,
                       "GBps": am_gbs, "hbm_frac": am_gbs / hbm_peak, "hbm_frac_nominal_8TBps": am_gbs / 8000.0,
                       "algorithmic_bytes_per_sample": am_bytes,
                       "note": "config[3], secondary; not part of `value`"},
            },
            "ingest": ingest,
            "parity": parity,
            "cpu_baseline": cpu,
        }
        if config4 is not None:
            line["config4_single_gpu"] = config4
        if split is not None:
            line["split_capture"] = split
        print(json.dumps(line))
    sdr_other.close()
    sdr.close()
    if world > 1:
        dist.barrier()   # rank 0 also ran the ingest probe; leave together
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
