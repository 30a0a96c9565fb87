"""Every launch-plan regime of the batched and streaming kernels against the float64 golden model.

csrc/plan.h cuts each capture into work in a different way for each kernel, and the kernel code that differs
between regimes is where indexing bugs live: the spectrum's frames per warp, empty warps in the last unit, the
64-frame cap and the separate finalize with a carried spectrum; the FP32 FIR segments with their pre-roll tile,
a ragged last chunk or tile and a last segment of one tile; the tensor-core engine's cp.async tile inside a
segment that starts with a pre-roll, and several rounds of work items per CTA; the wave loop of
b200sdr_batch_host.  The shapes here are chosen from the plan, not from the signal.
test_plan_regimes_at_148_sms pins every shape to its regime on the CPU, so a change to plan.h that moves a
shape out of its regime fails there instead of quietly emptying the coverage, and each GPU test asserts the
same regime with the device's own SM count, so a part with another SM count fails instead of testing
something else.

Tolerances are those of test_gpu_parity.py (BASELINE.json north_star).
"""
import ctypes as C
import functools
import os
import subprocess
import tempfile

import numpy as np
import pytest

from oracle_api import (AVG_EMA, AVG_MEAN, SYNTH_AM, SYNTH_MULTITONE, SYNTH_WBFM, WIN_BLACKMAN, WIN_RECT, Golden,
                        wrap_phase)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B200_SMS = 148

SPEC_RTOL = 1e-5      # relative, per bin
DISC_ATOL = 1e-4      # radians
FM_AUDIO_ATOL = 1e-4 * 240000.0 / (2 * np.pi * 75000.0)
AM_AUDIO_ATOL = 1e-6  # AM audio is O(0.05); fp32 FIRs give ~1e-8
# tensor-core engine against the FP32 engine (test_gpu_parity.test_tensor_engine_golden_fixture_and_engines_agree);
# the first discriminator outputs see the filter's rise from x[n < 0] = 0 and are left out
TC_VS_FP32_AUDIO, TC_VS_FP32_DISC, TC_VS_FP32_SKIP = 2e-6, 5e-6, 8

WAVE_BYTES = 192 << 20  # kWaveBytes of csrc/api.cu: input bytes per wave of b200sdr_batch_host


def ceil_div(a, b):
    return -(-a // b)


# ------------------------------------------------------------------------------------------- plans
@functools.lru_cache(maxsize=None)
def _plan_functions():
    """emu_plan_spectrum of the emulation harness (built by conftest.py) and the FIR plans of tests/emu/emu_plans.cpp,
    compiled into a temporary directory because the tree may be read-only"""
    kernels = C.CDLL(os.path.join(ROOT, "tests", "emu", "libemu_kernels.so"))
    with tempfile.TemporaryDirectory() as tmp:
        so = os.path.join(tmp, "libemu_plans.so")
        subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", so,
                        os.path.join(ROOT, "tests", "emu", "emu_plans.cpp")], check=True)
        plans = C.CDLL(so)  # stays mapped once the directory is gone
    fns = {"emu_plan_spectrum": kernels.emu_plan_spectrum, "emu_plan_wbfm": plans.emu_plan_wbfm,
           "emu_plan_wbfm_tc": plans.emu_plan_wbfm_tc, "emu_plan_am": plans.emu_plan_am}
    for fn in fns.values():
        fn.argtypes = [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
    return fns


def _plan(name, n_out, len_bytes, n_captures, sms):
    out = (C.c_uint32 * n_out)()
    _plan_functions()[name](len_bytes, n_captures, sms, out)
    return list(out)


def spectrum_regime(len_bytes, n_captures, sms):
    frames, fpw, units, grid = _plan("emu_plan_spectrum", 4, len_bytes, n_captures, sms)
    last = frames - (units - 1) * 4 * fpw
    return dict(frames=frames, fpw=fpw, units=units, grid=grid, len_mod16=len_bytes % 16,
                fpw_capped=ceil_div(frames, 2 * 148 * 4) > fpw,
                last_unit_frames=last, empty_warps_last_unit=4 - ceil_div(last, fpw),
                tail_bytes=len_bytes - 2 * (512 * (frames - 1) + 1024),
                more_units_than_grid=units * n_captures > grid,
                # launch_spectrum folds the finalize into the last CTA only for one capture of <= 128 units
                separate_finalize=not (n_captures == 1 and units <= 128))


def _segments(tiles, chunks, tps, segments, len_bytes):
    return dict(tiles=tiles, segments=segments, last_segment_tiles=tiles - (segments - 1) * tps,
                ragged_chunk=(len_bytes // 2) % 200 != 0,  # B200_FM_CHUNK = B200_AM_CHUNK = 200 samples
                ragged_tile=chunks % 128 != 0)             # 128 chunks (threads) per tile


def wbfm_regime(len_bytes, n_captures, sms):
    return _segments(*_plan("emu_plan_wbfm", 4, len_bytes, n_captures, sms), len_bytes)


def am_regime(len_bytes, n_captures, sms):
    tiles, chunks, tps, segments, q_count = _plan("emu_plan_am", 5, len_bytes, n_captures, sms)
    # k_am_back scans the envelope in tiles of 4096 samples
    return dict(_segments(tiles, chunks, tps, segments, len_bytes), q_count=q_count, back_tiles=ceil_div(q_count, 4096))


def tc_regime(len_bytes, n_captures, sms):
    tiles, rows, tps, segments, grid = _plan("emu_plan_wbfm_tc", 5, len_bytes, n_captures, sms)
    items = segments * n_captures
    r = dict(tiles=tiles, segments=segments, items=items, rounds=ceil_div(items, grid), ragged_row=len_bytes % 320 != 0)
    if r["ragged_row"]:  # launch_wbfm_tc_batch: the tile with the ragged last row is filled by cp.async, not TMA
        r["cp_async_tile_segment"] = (len_bytes // 320 // 125) // tps
    return r


def wave_regime(len_bytes, n_captures, sms):
    per_wave = max(1, min(WAVE_BYTES // len_bytes, n_captures))
    return dict(waves=[min(per_wave, n_captures - c) for c in range(0, n_captures, per_wave)])


def stream_cuts(slot_bytes):
    """a stream of three and a half ring slots, cut into blocks at random 4-byte boundaries"""
    total = 3 * slot_bytes + (2 * slot_bytes // 5) // 4 * 4
    return random_cuts(total, 65536, 140)


def stream_regime(slot_bytes, _n_captures, sms):
    """the spectrum launches of the streaming path for stream_cuts(slot_bytes): process_samples appends blocks to the
    open slot and submits it when full or when the next block does not fit; each launch runs over the unread
    512-sample overlap of the last one plus the slot's bytes"""
    slots, pending = [], 0
    for n in stream_cuts(slot_bytes):
        if pending + n > slot_bytes:
            slots.append(pending)
            pending = 0
        pending += n
        if pending >= slot_bytes:
            slots.append(pending)
            pending = 0
    slots.append(pending)  # submitted by get_spectrum
    launches, left = [], 0
    for s in slots:
        r = spectrum_regime(left + s, 1, sms)
        launches.append(r)
        left += s - 1024 * r["frames"]
    sep = [r for r in launches if r["separate_finalize"]]
    return dict(launches=len(launches), separate_finalize_launches=len(sep), separate_finalize_fpw=sorted({r["fpw"] for r in sep}))


REGIME_OF = {"spectrum": spectrum_regime, "wbfm": wbfm_regime, "am": am_regime, "tc": tc_regime, "waves": wave_regime,
             "stream": stream_regime}

# a. spectrum frames per warp: 4 bytes after the last frame, and the last unit holds one frame (three empty warps)
SPEC_FPW = {2: (1_214_468, 149), 5: (4_855_812, 238), 17: (19_429_380, 280), 41: (48_535_556, 290), 64: (76_548_100, 293)}
SPEC_CAP_LEN = 2 * (1024 + 512 * 100_000) + 1020
# c. captures of 4, 8 and 12 bytes mod 16
UNALIGNED = [(3, 262_148), (4, 1_214_472), (5, 600_076)]
# e. FP32 WBFM and AM
FP32_SHAPES = [(819_216, 1), (871_616, 1), (1_689_616, 2), (4_800_016, 7), (1_638_400, 1), (1_638_800, 1), (3_277_200, 1)]
# f. tensor-core WBFM
TC_SHAPES = [(4_800_016, 1), (360_016, 37), (2_400_016, 40), (1_600_016, 150)]
# g. b200sdr_batch_host
WAVE_LEN = (64 << 20) + 16

# name -> [(plan, len_bytes (slot_bytes for "stream"), n_captures, the fields that make the regime)]
REGIMES = {
    **{f"spectrum_fpw{fpw}": [("spectrum", n, 1, dict(fpw=fpw, units=u, last_unit_frames=1, empty_warps_last_unit=3,
                                                       tail_bytes=4, separate_finalize=True))]
       for fpw, (n, u) in SPEC_FPW.items()},
    "spectrum_fpw_cap": [("spectrum", SPEC_CAP_LEN, 3, dict(frames=100_001, fpw=64, fpw_capped=True, units=391, grid=296,
                                                           more_units_than_grid=True, tail_bytes=1020))],
    "spectrum_unaligned_3": [("spectrum", 262_148, 3, dict(len_mod16=4, fpw=1, separate_finalize=True)),
                             ("spectrum", 262_148, 1, dict(separate_finalize=False))],
    "spectrum_unaligned_4": [("spectrum", 1_214_472, 4, dict(len_mod16=8, fpw=2, separate_finalize=True))],
    "spectrum_unaligned_5": [("spectrum", 600_076, 5, dict(len_mod16=12, fpw=1, separate_finalize=True))],
    "stream_1MiB": [("stream", 1 << 20, None, dict(launches=4, separate_finalize_launches=3, separate_finalize_fpw=[1]))],
    "stream_4MiB": [("stream", 1 << 22, None, dict(launches=4, separate_finalize_launches=4, separate_finalize_fpw=[2, 4]))],
    "fp32_819216x1": [("wbfm", 819_216, 1, dict(tiles=17, segments=2, last_segment_tiles=1, ragged_chunk=True)),
                      ("am", 819_216, 1, dict(segments=2, last_segment_tiles=1, q_count=2049))],
    "fp32_871616x1": [("wbfm", 871_616, 1, dict(segments=2, last_segment_tiles=2, ragged_chunk=True, ragged_tile=True)),
                      ("am", 871_616, 1, dict(segments=2, ragged_chunk=True, ragged_tile=True))],
    "fp32_1689616x2": [("wbfm", 1_689_616, 2, dict(segments=3, last_segment_tiles=2, ragged_chunk=True, ragged_tile=True)),
                       ("am", 1_689_616, 2, dict(segments=3, ragged_chunk=True))],
    "fp32_4800016x7": [("wbfm", 4_800_016, 7, dict(segments=6, ragged_chunk=True, ragged_tile=True)),
                       ("am", 4_800_016, 7, dict(segments=6, ragged_chunk=True, back_tiles=3))],
    "fp32_1638400x1": [("am", 1_638_400, 1, dict(q_count=4096, back_tiles=1, segments=2, ragged_tile=False))],
    "fp32_1638800x1": [("am", 1_638_800, 1, dict(q_count=4097, back_tiles=2, segments=3, last_segment_tiles=1)),
                       ("wbfm", 1_638_800, 1, dict(segments=3, last_segment_tiles=1))],
    "fp32_3277200x1": [("am", 3_277_200, 1, dict(q_count=8193, back_tiles=3, segments=5, last_segment_tiles=1)),
                       ("wbfm", 3_277_200, 1, dict(segments=5, last_segment_tiles=1))],
    "tc_4800016x1": [("tc", 4_800_016, 1, dict(segments=16, rounds=1, ragged_row=True, cp_async_tile_segment=15))],
    "tc_360016x37": [("tc", 360_016, 37, dict(segments=2, items=74, rounds=1, ragged_row=True, cp_async_tile_segment=1))],
    "tc_2400016x40": [("tc", 2_400_016, 40, dict(segments=7, rounds=2, ragged_row=True, cp_async_tile_segment=6))],
    "tc_1600016x150": [("tc", 1_600_016, 150, dict(segments=5, items=750, rounds=6, ragged_row=True, cp_async_tile_segment=4))],
    # waves of 2 and 1 captures: the plans of the last wave are those of one capture
    "waves": [("waves", WAVE_LEN, 3, dict(waves=[2, 1])),
              ("spectrum", WAVE_LEN, 2, dict(more_units_than_grid=True)),
              ("wbfm", WAVE_LEN, 2, dict(ragged_chunk=True, ragged_tile=True)),
              ("tc", WAVE_LEN, 2, dict(segments=73, ragged_row=True)),
              ("tc", WAVE_LEN, 1, dict(segments=140)),
              ("tc", WAVE_LEN, 3, dict(segments=48))],
}


def assert_regime(name, sms):
    for kind, len_bytes, n_captures, want in REGIMES[name]:
        got = REGIME_OF[kind](len_bytes, n_captures, sms)
        moved = {k: (got[k], v) for k, v in want.items() if got[k] != v}
        assert not moved, f"{name}: {kind} plan of {n_captures} x {len_bytes} bytes at {sms} SMs (got, intended): {moved}"


@pytest.mark.parametrize("name", sorted(REGIMES))
def test_plan_regimes_at_148_sms(name):
    """csrc/plan.h (through the emulation harness) still puts every shape the GPU tests below use in its regime"""
    assert_regime(name, B200_SMS)


# ------------------------------------------------------------------------------------------ checks
def spec_check(out, gold, rtol=SPEC_RTOL):
    rel = np.abs(out.astype(np.float64) - gold) / gold
    assert rel.max() <= rtol, f"max rel err {rel.max():.3e} at bin {rel.argmax()}"


def spec_check_few_frames(out, gold):
    """eps * sqrt(P_k * P_max) bound where few frames are averaged (see test_gpu_parity.spec_check_few_frames)"""
    err = np.abs(out.astype(np.float64) - gold)
    bound = 1e-5 * gold + 4e-7 * np.sqrt(gold * gold.max())
    assert np.all(err <= bound), f"worst excess {np.max(err / bound):.2f}x at bin {np.argmax(err / bound)}"


def spec_check_window(out, gold):
    """as test_gpu_parity.test_spectrum_other_windows: RECT and Blackman leave bins far below the strongest"""
    rel = np.abs(out.astype(np.float64) - gold) / np.maximum(gold, 1e-7 * gold.max())
    assert rel.max() <= SPEC_RTOL, f"max rel err {rel.max():.3e} at bin {rel.argmax()}"


def wbfm_check(audio, disc, iq, g):
    ga, gd = g.wbfm(iq, want_disc=True)
    assert audio.size == ga.size and disc.size == gd.size
    assert np.max(np.abs(wrap_phase(disc - gd))) <= DISC_ATOL
    assert np.max(np.abs(audio - ga)) <= FM_AUDIO_ATOL


def am_check(audio, iq, g):
    ga = g.am(iq)
    assert audio.size == ga.size and np.max(np.abs(audio - ga)) <= AM_AUDIO_ATOL


def random_cuts(total, max_block, seed):
    rng = np.random.default_rng(seed)
    cuts, left = [], total
    while left:
        n = int(min(left, 4 * rng.integers(1, max_block // 4 + 1)))
        cuts.append(n)
        left -= n
    return cuts


def feed(s, iq, cuts):
    pos = 0
    for n in cuts:
        while s.process_samples(iq[pos:pos + n], allow_busy=True) == 1:  # BUSY: ring full, call again
            s.sync()
        pos += n
    assert pos == iq.size


def dev_spectrum(s, iq, n_captures, len_each, offset=0):
    """b200sdr_batch_spectrum_dev over captures that start `offset` bytes into a fresh (256-byte aligned) allocation"""
    d_iq, d_out = s.dev_alloc(offset + iq.size), s.dev_alloc(4 * 1024 * n_captures)
    try:
        s.to_dev(d_iq + offset, iq)
        s.batch_spectrum_dev(d_iq + offset, n_captures, len_each, d_out)
        s.sync()
        return s.to_host(d_out, 4 * 1024 * n_captures, np.float32).reshape(n_captures, 1024)
    finally:
        s.dev_free(d_iq)
        s.dev_free(d_out)


def dev_all_chains(s, iq, n_captures, len_each):
    """spectrum, WBFM audio and AM audio of the batch through the three _dev entry points"""
    na, nam = s.lib.b200sdr_wbfm_audio_len(len_each), s.lib.b200sdr_am_audio_len(len_each)
    d_iq = s.dev_alloc(iq.size)
    d_spec, d_fm, d_am = (s.dev_alloc(4 * k * n_captures) for k in (1024, na, nam))
    try:
        s.to_dev(d_iq, iq)
        s.batch_spectrum_dev(d_iq, n_captures, len_each, d_spec)
        s.batch_wbfm_dev(d_iq, n_captures, len_each, d_fm)
        s.batch_am_dev(d_iq, n_captures, len_each, d_am)
        s.sync()
        return tuple(s.to_host(d, 4 * k * n_captures, np.float32).reshape(n_captures, k)
                     for d, k in ((d_spec, 1024), (d_fm, na), (d_am, nam)))
    finally:
        for d in (d_iq, d_spec, d_fm, d_am):
            s.dev_free(d)


@pytest.fixture(scope="module")
def g():
    return Golden()


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def sdr(sdr_lib):
    s = sdr_lib.B200Sdr()
    yield s
    s.close()


@pytest.fixture(scope="module")
def sdr_tc(sdr_lib):
    s = sdr_lib.B200Sdr(fir_engine=sdr_lib.FIR_ENGINE_TENSOR)
    yield s
    s.close()


# --------------------------------------------------------------------------------- a. frames per warp
@pytest.mark.gpu
@pytest.mark.parametrize("fpw", sorted(SPEC_FPW))
def test_spectrum_frames_per_warp(sdr, g, sms, fpw):
    assert_regime(f"spectrum_fpw{fpw}", sms)
    len_each = SPEC_FPW[fpw][0]
    iq = g.synth(1, len_each, SYNTH_MULTITONE, 100 + fpw)
    spec_check(dev_spectrum(sdr, iq, 1, len_each)[0], g.spectrum(iq)[0])


@pytest.mark.gpu
def test_spectrum_frames_per_warp_cap_in_a_batch(sdr, g, sms):
    """fpw capped at 64, and more units than the persistent grid has CTA slots"""
    assert_regime("spectrum_fpw_cap", sms)
    L = SPEC_CAP_LEN
    iq = g.synth(3, L, SYNTH_MULTITONE, 110)
    out = dev_spectrum(sdr, iq, 3, L)
    spec_check(out[0], g.spectrum(iq[:L])[0])
    for c in (1, 2):
        assert np.array_equal(out[c], dev_spectrum(sdr, iq[c * L:(c + 1) * L], 1, L)[0]), c


# ---------------------------------------------------------------------- b. EMA and windows across units
@pytest.mark.gpu
@pytest.mark.parametrize("beta", [0.1, 0.01])
@pytest.mark.parametrize("fpw", [5, 17])
def test_spectrum_ema_across_units(sdr_lib, g, sms, fpw, beta):
    """the EMA weight beta (1 - beta)^(frames - 1 - m) over multi-frame warps in many units (~2 / beta frames count)"""
    assert_regime(f"spectrum_fpw{fpw}", sms)
    len_each = SPEC_FPW[fpw][0]
    iq = g.synth(1, len_each, SYNTH_MULTITONE, 120 + fpw)
    with sdr_lib.B200Sdr(chains=sdr_lib.CHAIN_SPECTRUM, avg_mode=AVG_EMA, ema_beta=beta) as s:
        out = dev_spectrum(s, iq, 1, len_each)[0]
    spec_check_few_frames(out, g.spectrum(iq, avg_mode=AVG_EMA, beta=beta)[0])


@pytest.mark.gpu
@pytest.mark.parametrize("window", [WIN_RECT, WIN_BLACKMAN], ids=["rect", "blackman"])
def test_spectrum_windows_across_units(sdr_lib, g, sms, window):
    assert_regime("spectrum_fpw5", sms)
    len_each = SPEC_FPW[5][0]
    iq = g.synth(1, len_each, SYNTH_MULTITONE, 130)
    with sdr_lib.B200Sdr(chains=sdr_lib.CHAIN_SPECTRUM, window=window) as s:
        out = dev_spectrum(s, iq, 1, len_each)[0]
    spec_check_window(out, g.spectrum(iq, window=window)[0])


# ---------------------------------------------------------------------------- c. unaligned captures
@pytest.mark.gpu
@pytest.mark.parametrize("offset", [0, 2])
@pytest.mark.parametrize("n_captures,len_each", UNALIGNED)
def test_spectrum_unaligned_captures(sdr, g, sms, n_captures, len_each, offset):
    """b200sdr_batch_spectrum_dev takes lengths that are a multiple of 4 and 2-byte aligned pointers: captures start at
    every residue mod 16.  The summation tree depends on the length only, so each capture must equal, bit for bit,
    the same bytes run alone from an aligned buffer."""
    assert_regime(f"spectrum_unaligned_{n_captures}", sms)
    iq = g.synth(n_captures, len_each, SYNTH_MULTITONE, 140 + n_captures)
    out = dev_spectrum(sdr, iq, n_captures, len_each, offset)
    for c in range(n_captures):
        cap = iq[c * len_each:(c + 1) * len_each]
        spec_check(out[c], g.spectrum(cap)[0])
        assert np.array_equal(out[c], dev_spectrum(sdr, cap, 1, len_each)[0]), c


# ------------------------------------------------------------- d. streaming spectrum, separate finalize
@pytest.mark.gpu
@pytest.mark.parametrize("avg_mode", [AVG_MEAN, AVG_EMA], ids=["mean", "ema"])
@pytest.mark.parametrize("slot_bytes", [1 << 20, 1 << 22], ids=["1MiB", "4MiB"])
def test_streaming_spectrum_large_slots(sdr_lib, g, sms, slot_bytes, avg_mode):
    """slots of more than 128 units go through k_spectrum_finalize, which adds the spectrum carried from the slots
    before (scaled by (1 - beta)^frames for EMA)"""
    assert_regime(f"stream_{slot_bytes >> 20}MiB", sms)
    cuts = stream_cuts(slot_bytes)
    iq = g.synth(1, sum(cuts), SYNTH_MULTITONE, 150)
    with sdr_lib.B200Sdr(chains=sdr_lib.CHAIN_SPECTRUM, slot_bytes=slot_bytes, ring_slots=4, avg_mode=avg_mode,
                         ema_beta=0.1) as s:
        feed(s, iq, cuts)
        spec, frames = s.get_spectrum()
    gold, gold_frames = g.spectrum(iq, avg_mode=avg_mode, beta=0.1)
    assert frames == gold_frames
    spec_check(spec, gold) if avg_mode == AVG_MEAN else spec_check_few_frames(spec, gold)


# ------------------------------------------------------------------- e. FP32 WBFM and AM, segmented
@pytest.mark.gpu
@pytest.mark.parametrize("len_each,n_captures", FP32_SHAPES)
def test_fp32_fir_chains_segmented_and_ragged(sdr, g, sms, len_each, n_captures):
    assert_regime(f"fp32_{len_each}x{n_captures}", sms)
    iq = g.synth(n_captures, len_each, SYNTH_WBFM, 160)
    audio, disc = sdr.wbfm(iq, n_captures, want_disc=True)
    iq_am = g.synth(n_captures, len_each, SYNTH_AM, 170)
    am = sdr.am(iq_am, n_captures)
    for c in range(n_captures):
        part = slice(c * len_each, (c + 1) * len_each)
        wbfm_check(audio[c], disc[c], iq[part], g)
        am_check(am[c], iq_am[part], g)


# -------------------------------------------------------------- f. tensor-core WBFM, segmented
@pytest.mark.gpu
@pytest.mark.parametrize("len_each,n_captures", TC_SHAPES)
def test_tensor_engine_segmented_and_ragged(sdr, sdr_tc, g, sms, len_each, n_captures):
    """every capture against the FP32 engine; the first, the last and three seeded picks against the golden model"""
    assert_regime(f"tc_{len_each}x{n_captures}", sms)
    iq = g.synth(n_captures, len_each, SYNTH_WBFM, 180)
    audio, disc = sdr_tc.wbfm(iq, n_captures, want_disc=True)
    a32, d32 = sdr.wbfm(iq, n_captures, want_disc=True)
    assert np.max(np.abs(audio - a32)) <= TC_VS_FP32_AUDIO
    assert np.max(np.abs(wrap_phase(disc - d32))[:, TC_VS_FP32_SKIP:]) <= TC_VS_FP32_DISC
    picks = {0, n_captures - 1} | set(np.random.default_rng(n_captures).integers(0, n_captures, 3).tolist())
    for c in sorted(picks):
        wbfm_check(audio[c], disc[c], iq[c * len_each:(c + 1) * len_each], g)


# ------------------------------------------------------------------------ g. batch_host across waves
@pytest.mark.gpu
@pytest.mark.parametrize("engine", ["fp32", "tensor"])
def test_batch_host_across_waves(sdr_lib, g, sms, engine):
    """three captures of 64 MiB + 16 bytes run as waves of two and one through the double-buffered wave loop; each
    capture's results equal those of the _dev entry points on the whole batch at once"""
    assert_regime("waves", sms)
    L, n = WAVE_LEN, 3
    kinds = (SYNTH_MULTITONE, SYNTH_WBFM, SYNTH_AM)
    iq = np.concatenate([g.synth(1, L, kinds[c], 190 + c) for c in range(n)])
    fir = sdr_lib.FIR_ENGINE_TENSOR if engine == "tensor" else sdr_lib.FIR_ENGINE_FP32
    with sdr_lib.B200Sdr(fir_engine=fir) as s:
        spec = np.empty((n, 1024), np.float32)
        fm = np.empty((n, sdr_lib.wbfm_audio_len(L)), np.float32)
        am = np.empty((n, sdr_lib.am_audio_len(L)), np.float32)
        s.batch_host(sdr_lib.CHAIN_SPECTRUM | sdr_lib.CHAIN_WBFM | sdr_lib.CHAIN_AM, iq, n, L, spectrum=spec, wbfm=fm, am=am)
        d_spec, d_fm, d_am = dev_all_chains(s, iq, n, L)
    assert np.array_equal(spec, d_spec) and np.array_equal(am, d_am)
    if engine == "fp32":
        assert np.array_equal(fm, d_fm)
    else:  # the tensor engine's segments follow the number of captures in the launch
        assert np.max(np.abs(fm - d_fm)) <= 1e-6
    for c in (0, 2):  # one capture of each wave
        cap = iq[c * L:(c + 1) * L]
        spec_check(spec[c], g.spectrum(cap)[0])
        assert np.max(np.abs(fm[c] - g.wbfm(cap))) <= FM_AUDIO_ATOL
        am_check(am[c], cap, g)
