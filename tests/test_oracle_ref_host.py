"""Oracle A: the reference's own, UNMODIFIED sample-transfer C (oracle/_ref, compiled by oracle/Makefile from
the reference's source tree, which this repository does not contain) -- and our restatement of it checked
against it.  CPU only.  SURVEY.md section 4 KATs / section 8c.

What the reference's USB_ReadPacket returns is also stored in tests/golden/reference_vectors.npz, so the
restatement is checked against it without the reference's sources; the class FSM tests need oracle A."""
import os
import re

import numpy as np
import pytest

from oracle_api import ROOT, SYNTH_COUNTER, Golden, RefHost

ref = RefHost()
needs_ref = pytest.mark.skipif(not ref.available,
                               reason="needs oracle A: build it with REF=<the reference's source tree> make -C oracle")
REF = np.load(os.path.join(ROOT, "tests", "golden", "reference_vectors.npz"))


@pytest.fixture(scope="module")
def g():
    return Golden()


def test_usb_readpacket_is_word_granular(g):
    # KAT: len = 510 -> 128 words = 512 bytes written, first 510 identical (usbh_rtlsdr.h:256-261 warning)
    src = (np.arange(600) * 7 + 3).astype(np.uint8)
    for copy in [g.ingest_copy] + ([ref.read_packet] if ref.available else []):
        dest, written = copy(src, 510)
        assert written == 512
        assert np.array_equal(dest[:512], src[:512])
        assert np.all(dest[512:] == 0xEE)


@pytest.mark.parametrize("length", [0, 1, 2, 3, 4, 5, 63, 64, 509, 510, 511, 512])
def test_restated_copy_matches_reference(g, length):
    src = np.random.default_rng(length).integers(0, 256, 600, dtype=np.uint8)
    d_ref, w_ref = REF[f"copy_dest_{length}"], int(REF["copy_written"][list(REF["copy_lengths"]).index(length)])
    if ref.available:
        d_live, w_live = ref.read_packet(src, length)
        assert w_live == w_ref and np.array_equal(d_live, d_ref)
    d_gold, w_gold = g.ingest_copy(src, length)
    assert w_ref == w_gold == 4 * ((length + 3) // 4)
    assert np.array_equal(d_ref, d_gold)


@needs_ref
def test_class_fsm_cadence_and_buffer(tmp_path, g):
    # 5 full URBs of the live buffSize (512, usbh_rtlsdr.c:230) of the test-mode counter stream
    data = g.synth(1, 512 * 5, SYNTH_COUNTER, 0)
    out, log = ref.run_stream(data, 512, 7, str(tmp_path))
    assert np.array_equal(out, data)  # bytes arrive unchanged, in order
    init = re.search(r"REF_INIT status=(\d+) buff=(0x[0-9a-f]+) size=(\d+) ep=(0x[0-9a-f]+) mps=(\d+) prescaler=(\d+)", log)
    assert init and init.group(1) == "0"
    assert int(init.group(2), 16) == 0xC007F800  # LCD_FB_START_ADDRESS + 480*272*4 (usbh_rtlsdr.c:227)
    assert (int(init.group(3)), int(init.group(4), 16), int(init.group(5))) == (512, 0x81, 512)
    assert int(init.group(6)) == 200000000 // 2 // 100000 - 1  # TIM5 at 100 kHz (usbh_rtlsdr.c:237)
    summ = re.search(r"REF_SUMMARY blocks=(\d+) submits=(\d+) polls_min=(\d+) polls_max=(\d+) .* final_state=(\d+)", log)
    assert summ
    blocks, submits, pmin, pmax, final = map(int, summ.groups())
    assert blocks == 5 and submits == 5      # exactly one URB per block
    assert pmin == pmax == 3                 # START -> WAIT -> COMPLETE -> START
    assert final == 0                        # RTLSDR_XFER_START
    # the reference's own throughput log line: bytes*100/CNT kB/s with CNT = 7
    assert log.count("Xfer complete 512 B, 7314 kB/s") == 5


@needs_ref
def test_stream_with_short_last_urb(tmp_path):
    data = np.random.default_rng(3).integers(0, 256, 512 * 3 + 200, dtype=np.uint8)
    out, log = ref.run_stream(data, 512, 11, str(tmp_path))
    assert np.array_equal(out, data)
    assert "Xfer complete 200 B" in log


@needs_ref
def test_large_urbs_use_multiple_packets(tmp_path):
    # 127 x 512 = 65024 bytes: the largest block one URB can carry (uint16_t length, usbh_ioreq.c:220)
    data = np.random.default_rng(4).integers(0, 256, 65024 * 2, dtype=np.uint8)
    out, log = ref.run_stream(data, 65024, 100, str(tmp_path))
    assert np.array_equal(out, data)
    assert log.count("Xfer complete 65024 B") == 2
