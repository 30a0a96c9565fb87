"""SURVEY.md section 5: compute-sanitizer over the device kernels.  One subprocess per tool runs the
smoke path plus a streaming block through every chain; any memcheck error, shared-memory race or
barrier misuse fails the test."""
import os
import shutil
import subprocess
import sys
import textwrap

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = textwrap.dedent("""
    import importlib, sys
    import numpy as np
    sys.path.insert(0, %r)
    pkg = importlib.import_module("stm32f7-rtlsdr_b200")
    iq = pkg.synth_fill_host(2, 61440 * 2 + 4800, pkg.SYNTH_WBFM, 3)          # > 1 tile per capture, ragged tail
    with pkg.B200Sdr(slot_bytes=65024, ring_slots=3) as s:
        s.spectrum(iq, 2); s.wbfm(iq, 2); s.am(iq, 2); s.convert_cf32(iq[:4096], pkg.WINDOW_HANN)
        for off in range(0, 65024 * 3, 65024):
            while s.process_samples(iq[off:off + 65024], allow_busy=True) == pkg.BUSY:
                s.sync()
        s.get_spectrum(); s.get_audio(pkg.CHAIN_WBFM); s.get_audio(pkg.CHAIN_AM)
        s.render_spectrum(None, 0.0, 100.0)
        s.render_waterfall(s.spectrum(iq[:65536 * 3], 3), 0.0, 100.0)
        # fused finalize + exchange kernel with a world of one (the sanitizer serialises kernels, so a
        # multi-rank wait cannot be run under it)
        s.exchange_create(1, 0); s.exchange_connect([b""])
        d_in, d_out = s.dev_alloc(65536), s.dev_alloc(4096)
        s.lib.b200sdr_copy_to_dev(s.ctx, d_in, iq.ctypes.data, 65536)
        s.split_spectrum_dev(d_in, 65536, 63, d_out); s.exchange_wait()
        s.dev_free(d_in); s.dev_free(d_out)
        # K0: ragged host block (head / tail words, last warps), then live blocks starting on odd word boundaries
        cnt = (np.arange(16384 + 2048 + 20) %% 256).astype(np.uint8)
        cnt[5000] ^= 1
        assert s.counter_check(cnt, 0)[0] == 2
    with pkg.B200Sdr(chains=pkg.CHAIN_COUNTER, slot_bytes=65024, ring_slots=3, submit_bytes=4) as c:
        for off in range(0, 4 * 4100, 4100):
            c.process_samples(cnt[off:off + 4100])
        assert c.get_counter_check()[0] == 2
    # tensor-core FIR engine (csrc/wbfm_tc.cuh): two full tiles through the TMA tensor map + a ragged one through the
    # bounds-checked cp.async fill per capture, mbarrier pipeline, tcgen05.mma / tcgen05.ld, named barrier of the epilogue
    iq2 = pkg.synth_fill_host(2, 40000 * 2 + 4800, pkg.SYNTH_WBFM, 3)
    with pkg.B200Sdr(chains=pkg.CHAIN_WBFM, fir_engine=pkg.FIR_ENGINE_TENSOR) as t:
        a = t.wbfm(iq2, 2)
        b, d = t.wbfm(iq2, 2, want_disc=True)
        assert np.array_equal(a, b) and np.isfinite(d).all()
    print("SANITIZED_RUN_OK")
""") % ROOT


@pytest.mark.parametrize("tool", ["memcheck", "racecheck", "synccheck"])
def test_compute_sanitizer_clean(tool, sdr_lib, tmp_path):
    cs = shutil.which("compute-sanitizer") or "/usr/local/cuda/bin/compute-sanitizer"
    if not os.access(cs, os.X_OK):
        pytest.skip("compute-sanitizer not installed or not executable by this user")
    script = tmp_path / "run.py"
    script.write_text(SCRIPT)
    try:
        res = subprocess.run([cs, "--tool", tool, "--error-exitcode", "9", sys.executable, str(script)],
                             capture_output=True, text=True, timeout=900)
    except PermissionError:
        pytest.skip("compute-sanitizer may not be executed by this user")
    tail = (res.stdout + res.stderr)[-3000:]
    assert res.returncode == 0, tail
    assert "SANITIZED_RUN_OK" in res.stdout, tail
    assert "ERROR SUMMARY: 0 errors" in tail or "0 hazards displayed (0 errors, 0 warnings)" in tail, tail
