"""SURVEY.md section 8f rows 2 and 4: the RTL2832 / E4000 front-end parameter math of the product
(include/b200sdr_frontend.h, host-only) against the reference's OWN routines compiled on the host
(oracle A: RTLSDR_set_sample_rate, RTLSDR_set_fir, E4K_compute_pll_params) -- bit-exact -- plus
the KATs of SURVEY section 4 that need no reference build.  CPU only.

The reference's answers are stored in tests/golden/reference_vectors.npz (inputs included, see
tests/golden/make_reference_vectors.py), so the comparison runs without the reference's sources; when
oracle A is built from them, the stored answers are checked against it as well."""
import importlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "oracle", "_ref", "ref_ingest_cli")
have_ref = os.path.exists(CLI)
REF = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))


@pytest.fixture(scope="module")
def b(sdr_lib):
    return importlib.import_module("stm32f7-rtlsdr_b200.binding")


def ref(*args):
    out = subprocess.run([CLI, *map(str, args)], capture_output=True, text=True, check=True).stdout
    return [l for l in out.splitlines() if l.startswith("REF_")][-1].split()[1:]


def test_kats_from_the_survey(b):
    # 240 kS/s (the rate the firmware programs, usbh_rtlsdr.c:898), 2.4 MS/s, 2.048 MS/s
    assert b.rtl_resampler(240000)[1:] == (0x0E000000, 0x1E000000, 240000.0)
    assert b.rtl_resampler(2400000) == (0, 0x03000000, 0x03000000, 2400000.0)
    assert b.rtl_resampler(2048000)[1] == 0x03840000
    rc, packed, coeff = b.rtl_fir_pack()
    assert rc == 0 and packed.hex() == "cadcd7d8e0f20e3506509c0d71111471741941a5"
    assert coeff[:3] == [-54, -36, -41] and coeff[-1] == 421


def test_unsupported_rates_are_reported(b):
    for rate in (225000, 300001, 900000, 3200001, 28125, 1):
        assert b.rtl_resampler(rate) == (3, 0, 0, 0.0)  # B200SDR_NOT_SUPPORTED, outputs zeroed
    for rate in (225001, 300000, 900001, 3200000):
        assert b.rtl_resampler(rate)[0] == 0


def test_fir_pack_range_check(b):
    c = [0] * 16
    c[3] = 128
    assert b.rtl_fir_pack(c)[0] == 3
    c[3] = 0
    c[9] = -2049
    assert b.rtl_fir_pack(c)[0] == 3


def test_resampler_bit_exact_against_reference(b):
    for rate, ratio_ref, applied_ref, real_ref in zip(REF["rates"], REF["rate_ratio"], REF["rate_applied"], REF["rate_real"]):
        rate = int(rate)
        rc, ratio, applied, real_rate = b.rtl_resampler(rate)
        if rc != 0:   # a rate the chip cannot take (300 001 .. 900 000): reported, outputs zeroed, nothing to compare
            assert 300000 < rate <= 900000 and (rc, ratio, applied, real_rate) == (3, 0, 0, 0.0)
            continue
        assert (ratio, applied) == (int(ratio_ref), int(applied_ref)), rate
        assert real_rate == float(real_ref), rate
        if have_ref:
            a, r, real = ref("--rate", rate)
            assert (int(a), int(r)) == (int(ratio_ref), int(applied_ref)), rate
            assert float(real) == float(real_ref), rate  # %.17g round-trips a double exactly


def test_fir_bytes_bit_exact_against_reference(b):
    assert b.rtl_fir_pack()[1] == REF["fir_bytes"].tobytes()
    if have_ref:
        assert ref("--fir")[0] == REF["fir_bytes"].tobytes().hex()


def test_e4k_pll_bit_exact_against_reference(b):
    for f, want_per_osc in zip(REF["pll_freqs"], REF["pll"]):
        for osc, want in zip(REF["pll_oscs"], want_per_osc):
            want = [int(v) for v in want]
            flo, fields = b.e4k_pll_params(int(osc), int(f))
            assert [flo, *fields] == want, (osc, f)
            if have_ref:
                assert [int(v) for v in ref("--e4k", osc, f)] == want, (osc, f)
    # invalid oscillator -> 0, like is_fosc_valid()
    assert b.e4k_pll_params(15999999, 100000000)[0] == 0
    if have_ref:
        assert int(ref("--e4k", 15999999, 100000000)[0]) == 0


def test_e4k_kat_at_the_firmware_frequency(b):
    flo, (fosc, want, got, x, z, r, r_idx, three) = b.e4k_pll_params(28800000, 99700000)
    assert (flo, got, x, z, r, r_idx, three) == (99699993, 99699993, 50972, 110, 32, 13, 1)


# ---- E4000 band / RF filter / IF bandwidth selection (tuner_e4k.c:218-277, :363-372, :871-878) ----

def test_e4k_band_thresholds(b):
    # E4K_tune_params state 4 (tuner_e4k.c:871-878): < 140 MHz VHF2, < 350 MHz VHF3, < 1135 MHz UHF, else L
    for hz, band in ((50000000, 0), (139999999, 0), (140000000, 1), (349999999, 1), (350000000, 2),
                     (1134999999, 2), (1135000000, 3), (2200000000, 3)):
        assert b.e4k_band(hz) == band, hz
    assert b.e4k_band(99699993) == 0  # the LO the firmware really gets for 99.7 MHz


def test_e4k_selection_kats(b):
    assert b.e4k_rf_filter(0, 99700000) == 0 and b.e4k_rf_filter(1, 200000000) == 0
    assert b.e4k_rf_filter(2, 433920000) == 3       # 425 MHz centre
    assert b.e4k_rf_filter(2, 370000000) == 0       # tie 360/380 -> first
    assert b.e4k_rf_filter(3, 1575420000) == 9      # GPS L1: 14.58 MHz from 1590, 15.42 from 1560
    assert b.e4k_rf_filter(7, 1575420000) == 0      # unknown band
    # the bandwidth the firmware asks for (RTLSDR_Handle->bw) against the three IF filters
    assert b.e4k_if_bw_index(0, 2400000) == (14, 2300000)
    assert b.e4k_if_bw_index(1, 2400000) == (26, 2400000)
    assert b.e4k_if_bw_index(2, 2400000) == (12, 2600000)
    assert b.e4k_if_bw_index(0, 27000000) == (0, 27000000)   # eight equal entries -> first
    assert b.e4k_if_bw_index(5, 2400000) == (0, 0)


def test_e4k_selection_bit_exact_against_reference(b):
    for band, want_row in zip(REF["rf_bands"], REF["rf_filter"]):
        for f, want in zip(REF["rf_freqs"], want_row):
            assert b.e4k_rf_filter(int(band), int(f)) == int(want), (band, f)
    for filt, idx_row, hz_row in zip(REF["ifbw_filters"], REF["ifbw_index"], REF["ifbw_selected_hz"]):
        for bw, idx, hz in zip(REF["ifbw_hz"], idx_row, hz_row):
            assert b.e4k_if_bw_index(int(filt), int(bw)) == (int(idx), int(hz)), (filt, bw)
    if not have_ref:
        return
    import ctypes as C
    lib = C.CDLL(os.path.join(ROOT, "oracle", "_ref", "libref_ingest.so"))
    lib.ref_e4k_rf_filter.argtypes = [C.c_int, C.c_uint32]
    lib.ref_e4k_if_bw_index.argtypes = [C.c_int, C.c_uint32]
    lib.ref_e4k_if_bw_hz.argtypes = [C.c_int, C.c_int]
    lib.ref_e4k_if_bw_hz.restype = C.c_uint32
    for band, want_row in zip(REF["rf_bands"], REF["rf_filter"]):
        for f, want in zip(REF["rf_freqs"], want_row):
            assert lib.ref_e4k_rf_filter(int(band), int(f)) == int(want), (band, f)
    for filt, idx_row, hz_row in zip(REF["ifbw_filters"], REF["ifbw_index"], REF["ifbw_selected_hz"]):
        for bw, idx, hz in zip(REF["ifbw_hz"], idx_row, hz_row):
            got = lib.ref_e4k_if_bw_index(int(filt), int(bw))
            assert (got, lib.ref_e4k_if_bw_hz(int(filt), got) if filt < 3 else 0) == (int(idx), int(hz)), (filt, bw)
    # the CLI agrees with the library (the path the other front-end tests use)
    assert ref("--e4k-rf", 2, 433920000) == ["3"]
    assert ref("--e4k-ifbw", 1, 2400000) == ["26", "2400000"]


# ------------------------------------------------------------ register initialisation sequence as data
def test_init_sequence_shape_and_errors(b):
    rc, n, raw = b.rtl_init_sequence()
    assert rc == 0 and n == 108 and len(raw) == 12 * 108
    rec = np.frombuffer(raw, np.dtype([("t", "u1"), ("r", "u1"), ("v", "<u2"), ("i", "<u2"), ("l", "<u2"), ("d", "u1", 2),
                                       ("step", "u1"), ("pad", "u1")]))
    assert set(rec["t"]) == {0x40, 0xC0} and not rec["r"].any() and set(rec["l"]) <= {1, 2}
    assert list(rec["step"]) == sorted(rec["step"]) and rec["step"][0] == 0 and rec["step"][-1] == 33
    # the resampler ratio of 240 kS/s (0x0E000000) travels high byte first in two 16-bit writes
    hi = rec[(rec["v"] == 0x9F20) & (rec["t"] == 0x40)][0]
    lo = rec[(rec["v"] == 0xA120) & (rec["t"] == 0x40)][0]
    assert bytes(hi["d"]) == b"\x0e\x00" and bytes(lo["d"]) == b"\x00\x00" and hi["l"] == 2
    # 2.4 MS/s: ratio 0x03000000; test mode off selects the demodulator output (0x05)
    rc, n, raw = b.rtl_init_sequence(2400000, flags=0)
    rec2 = np.frombuffer(raw, rec.dtype)
    assert rc == 0 and n == 108
    assert bytes(rec2[(rec2["v"] == 0x9F20) & (rec2["t"] == 0x40)][0]["d"]) == b"\x03\x00"
    assert rec2[(rec2["step"] == 31) & (rec2["t"] == 0x40)][0]["d"][0] == 0x05
    # capacity too small: count still reported, BUSY; unsupported rate / FIR: NOT_SUPPORTED and nothing emitted
    assert b.rtl_init_sequence(capacity=10)[:2] == (1, 108)
    assert b.rtl_init_sequence(capacity=0)[:2] == (1, 108)
    assert b.rtl_init_sequence(500000)[:2] == (3, 0)
    assert b.rtl_init_sequence(20000)[:2] == (3, 0)      # quotient would not fit 32 bits: rejected before the cast
    assert b.rtl_init_sequence(240000, fir=[4000] * 16)[:2] == (3, 0)
    assert b.rtl_init_sequence(0)[0] == 2


def test_init_sequence_bit_exact_against_reference(b, tmp_path):
    """The reference's own, unmodified USBH_RTLSDR_ClassRequest polled to completion in oracle A with a recording
    USBH_CtlReq: every setup packet and payload, in order, equals the product's list."""
    want = REF["init_trace"].tobytes()
    rc, n, got = b.rtl_init_sequence(240000, flags=1)
    assert rc == 0 and n == 108
    assert got == want
    if have_ref:
        path = str(tmp_path / "trace.bin")
        assert ref("--init-trace", path) == ["108"]
        assert open(path, "rb").read() == want


@pytest.mark.skipif(not have_ref, reason="needs oracle A: build it with REF=<the reference's source tree> make -C oracle")
def test_init_sequence_with_the_reference_tuner_driver_in_the_loop(b, tmp_path):
    """Same recording, but with the reference's own E4000 driver left in (Init, InitProcess, SetBW against a plain
    register-file model of the chip): its 70 I2C transfers land exactly where the product's list leaves room for
    the tuner (steps 29 and 30), and everything else is still the product's list, transfer for transfer."""
    path = str(tmp_path / "full.bin")
    assert ref("--init-trace-full", path)[0] == "178"
    dt = np.dtype([("t", "u1"), ("r", "u1"), ("v", "<u2"), ("i", "<u2"), ("l", "<u2"), ("d", "u1", 2), ("step", "u1"), ("pad", "u1")])
    full = np.fromfile(path, dt)
    tuner_i2c = np.flatnonzero(((full["i"] == 0x0610) | (full["i"] == 0x0600)) & (full["v"] == 0xC8))[2:]  # after the probe pair
    assert tuner_i2c.size == 70 and set(full["step"][tuner_i2c]) == {29, 30}
    keep = np.ones(full.size, bool)
    keep[tuner_i2c] = False
    assert full[keep].tobytes() == b.rtl_init_sequence(240000, flags=1)[2]


def test_fir_pack_round_trip_property(b):
    """property check (hypothesis): unpacking the 20 register bytes (8 x int8, then 4 x two int12 in three bytes) gives
    back every in-range coefficient set."""
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=200, deadline=None)
    @given(st.lists(st.integers(-128, 127), min_size=8, max_size=8), st.lists(st.integers(-2048, 2047), min_size=8, max_size=8))
    def check(c8, c12):
        rc, packed, _ = b.rtl_fir_pack(c8 + c12)
        assert rc == 0 and len(packed) == 20
        got8 = [v - 256 if v > 127 else v for v in packed[:8]]
        got12 = []
        for k in range(4):
            b0, b1, b2 = packed[8 + 3 * k: 11 + 3 * k]
            for v in ((b0 << 4) | (b1 >> 4), ((b1 & 0x0F) << 8) | b2):
                got12.append(v - 4096 if v > 2047 else v)
        assert got8 == c8 and got12 == c12

    check()
