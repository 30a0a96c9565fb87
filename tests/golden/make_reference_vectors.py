"""Regenerates tests/golden/reference_vectors.npz: what the original firmware's own routines return for
the inputs of tests/test_frontend_parity.py and tests/test_oracle_ref_host.py.

    python tests/golden/make_reference_vectors.py      (after __graft_entry__.build())

The original firmware's sources are not part of this repository, so the vectors are recorded through
the two implementations that were compared with those routines bit for bit while oracle A (oracle/_ref,
built by oracle/Makefile from the original's sources) was available: the product's front end
(include/b200sdr_frontend.h: RTLSDR_set_sample_rate, RTLSDR_set_fir, E4K_compute_pll_params, the E4000
filter selection, the ClassRequest control transfers) and oracle B's restatement of USB_ReadPacket
(oracle/golden.c).  Regenerate only at a commit whose tests pass against oracle A; whenever oracle A is
built, the tests compare these vectors with it again.  The inputs are stored beside the outputs, except the
copy sources, which are np.random.default_rng(length) bytes.
"""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle_api import Golden  # noqa: E402

COPY_LENGTHS = [0, 1, 2, 3, 4, 5, 63, 64, 509, 510, 511, 512]
E4K_CENTRES_MHZ = [360, 380, 405, 425, 450, 475, 505, 540, 575, 615, 670, 720, 760, 840, 890, 970,
                   1300, 1320, 1360, 1410, 1445, 1460, 1490, 1530, 1560, 1590, 1640, 1660, 1680, 1700, 1720, 1750]


def inputs():
    rates = [240000, 250000, 288000, 300000, 900001, 960000, 1024000, 1200000, 1400000, 1536000, 1800000, 1920000,
             2048000, 2400000, 2560000, 2880000, 3200000, 225001, 1000001, 2399999]
    rates += [int(x) for x in np.random.default_rng(0).integers(226000, 3200000, 40)]
    pll_freqs = [99700000,                       # the frequency the firmware tunes (tuner_e4k.c:1084)
                 52000000, 72399999, 72400000, 81200000, 108300000, 162500000, 216600000, 325000000, 350000000,
                 432000000, 667000000, 1199999999, 1200000000, 1700000000, 2200000000]
    pll_freqs += [int(x) for x in np.random.default_rng(1).integers(50_000_000, 2_200_000_000, 60)]
    rf_freqs = [0, 1, 0xFFFFFFFF, 360000000, 370000000, 369999999, 370000001, 1310000000, 1750000000]
    rf_freqs += [int(v) for v in np.random.default_rng(4).integers(50_000_000, 2_200_000_000, 3000)]
    for lo, hi in zip(E4K_CENTRES_MHZ, E4K_CENTRES_MHZ[1:]):   # every midpoint between centres, +-1 Hz (where the choice flips)
        mid = (lo + hi) * 500000
        rf_freqs += [mid - 1, mid, mid + 1]
    bws = [0, 1, 999999, 1000000, 2400000, 27000000, 0xFFFFFFFF] + list(range(900000, 28000000, 12500))
    return {"rates": np.array(rates, np.int64), "pll_oscs": np.array([28800000, 16000000, 30000000, 26000000], np.int64),
            "pll_freqs": np.array(pll_freqs, np.int64), "rf_bands": np.arange(5, dtype=np.int64),
            "rf_freqs": np.array(rf_freqs, np.int64), "ifbw_filters": np.arange(4, dtype=np.int64),
            "ifbw_hz": np.array(bws, np.int64), "copy_lengths": np.array(COPY_LENGTHS, np.int64)}


def copy_source(length):
    return np.random.default_rng(length).integers(0, 256, 600, dtype=np.uint8)


def main():
    b = importlib.import_module("stm32f7-rtlsdr_b200.binding")
    g = Golden()
    out = inputs()
    res = [b.rtl_resampler(int(r)) for r in out["rates"]]
    out["rate_status"] = np.array([r[0] for r in res], np.int64)
    out["rate_ratio"] = np.array([r[1] for r in res], np.int64)
    out["rate_applied"] = np.array([r[2] for r in res], np.int64)
    out["rate_real"] = np.array([r[3] for r in res], np.float64)
    out["fir_bytes"] = np.frombuffer(b.rtl_fir_pack()[1], np.uint8).copy()
    out["pll"] = np.array([[[flo, *fields] for flo, fields in (b.e4k_pll_params(int(o), int(f)) for o in out["pll_oscs"])]
                           for f in out["pll_freqs"]], np.int64)                       # [freq, osc, flo + 8 fields]
    out["rf_filter"] = np.array([[b.e4k_rf_filter(int(band), int(f)) for f in out["rf_freqs"]] for band in out["rf_bands"]], np.int64)
    ifbw = [[b.e4k_if_bw_index(int(filt), int(bw)) for bw in out["ifbw_hz"]] for filt in out["ifbw_filters"]]
    out["ifbw_index"] = np.array([[i for i, _ in row] for row in ifbw], np.int64)
    out["ifbw_selected_hz"] = np.array([[h for _, h in row] for row in ifbw], np.int64)
    rc, n, trace = b.rtl_init_sequence(240000, flags=1)
    assert rc == 0 and n == 108
    out["init_trace"] = np.frombuffer(trace, np.uint8).copy()
    written = []
    for length in COPY_LENGTHS:
        dest, w = g.ingest_copy(copy_source(length), length)
        out[f"copy_dest_{length}"] = dest
        written.append(w)
    out["copy_written"] = np.array(written, np.int64)
    path = os.path.join(ROOT, "tests", "golden", "reference_vectors.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "with", len(out), "arrays,", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
