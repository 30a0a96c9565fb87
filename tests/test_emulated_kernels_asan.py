"""The kernel source under the host emulation (tests/emu/emu_kernels.cpp) built with AddressSanitizer, on inputs and
outputs of EXACTLY their size: a kernel that reads past the end of a capture, or writes past the end of an output,
is reported here on the CPU.  On the GPU such a read only shows when the bytes after the capture change a result
(tests/test_gpu_footprint.py); here it is an error wherever it lands.

The child Python runs with libasan preloaded, so numpy's own buffers get redzones.  Each output must equal, bit for
bit, the regular emulation library's output on the same input padded with 64 zero bytes (the way
test_emulated_kernels.py calls it), which shows the padding is not needed.
"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "emu")


def _libasan():
    try:
        path = subprocess.run(["gcc", "-print-file-name=libasan.so"], capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        return None
    return path if os.path.isabs(path) and os.path.exists(path) else None


def test_emulated_kernels_read_and_write_only_their_buffers():
    asan = _libasan()
    if asan is None:
        pytest.skip("gcc has no libasan.so here")
    with tempfile.TemporaryDirectory() as tmp:  # the tree may be read-only
        so = os.path.join(tmp, "libemu_kernels_asan.so")
        subprocess.run(["g++", "-O1", "-g", "-fsanitize=address", "-fno-omit-frame-pointer", "-std=c++17", "-shared", "-fPIC",
                        "-o", so, os.path.join(EMU, "emu_kernels.cpp")], check=True)
        env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
        res = subprocess.run([sys.executable, os.path.abspath(__file__), so, os.path.join(EMU, "libemu_kernels.so")],
                             env=env, capture_output=True, text=True, timeout=900)
    assert "AddressSanitizer" not in res.stderr, res.stderr[-6000:]
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-6000:]
    assert "checked" in res.stdout, res.stdout


# ---------------------------------------------------------------------------------- the child process
def _load(path):
    e = C.CDLL(path)
    vp, u32, u64 = C.c_void_p, C.c_uint32, C.c_uint64
    e.emu_spectrum.argtypes = [vp, u32, u64, vp, u32, C.c_int, C.c_float, vp]
    e.emu_wbfm_batch.argtypes = [vp, u32, u64, u32, vp, vp]
    e.emu_wbfm_stream.argtypes = [vp, u32, u64, vp, vp, vp, vp, u32]
    e.emu_wbfm_tc_batch.argtypes = [vp, u32, u64, u32, vp, vp, vp, vp]
    e.emu_am_batch.argtypes = [vp, u32, u64, u32, vp, vp]
    e.emu_am_stream.argtypes = [vp, u32, u64, vp, vp, vp, vp, u32]
    e.emu_convert_cf32.argtypes = [vp, u64, vp, vp]
    e.emu_synth.argtypes = [vp, u32, u64, u32, u64, vp]
    e.emu_render_spectrum.argtypes = [vp, u32, C.c_float, C.c_float, C.c_float, vp]
    e.emu_render_waterfall.argtypes = [vp, u32, C.c_float, C.c_float, C.c_float, vp]
    e.emu_counter_check.argtypes = [vp, u64, C.c_int, C.POINTER(u64), C.POINTER(u64), vp, u64]
    return e


def _exact(a):
    """a copy in a buffer of its own, exactly a.nbytes long"""
    return np.array(a, copy=True, order="C")


def _padded(a):
    b = np.zeros(a.nbytes + 64, np.uint8)
    b[:a.nbytes] = np.ascontiguousarray(a).view(np.uint8).reshape(-1)
    return b


class _Pair:
    """one call on the ASan library with exact-size buffers and on the regular one with padded inputs"""

    def __init__(self, asan, plain):
        self.asan, self.plain, self.count = asan, plain, 0

    def __call__(self, name, inputs, outputs, args):
        """inputs: arrays; outputs: (count, dtype) pairs; args(ins, outs) -> the argument list of emu_<name>"""
        got = []
        for lib, prep in ((self.asan, _exact), (self.plain, _padded)):
            ins = [prep(a) for a in inputs]
            outs = [np.full(n, 0x7F if np.dtype(dt).kind == "u" else np.nan, dt) for n, dt in outputs]
            getattr(lib, "emu_" + name)(*args([a.ctypes.data for a in ins], [o.ctypes.data for o in outs]))
            got.append(outs)
        for i, (a, b) in enumerate(zip(*got)):
            assert a.view(np.uint8).tobytes() == b.view(np.uint8).tobytes(), f"{name}: output {i} differs from the padded run"
        self.count += 1
        return got[0]


def _synth_bytes(n, seed):
    return np.random.default_rng(seed).integers(0, 256, n, dtype=np.uint8)


def _child(asan_path, plain_path):
    run = _Pair(_load(asan_path), _load(plain_path))
    hann = (0.5 - 0.5 * np.cos(2 * np.pi * np.arange(1024) / 1024)).astype(np.float32)

    # spectrum: 4, 8 and 12 bytes after the last frame, one and three frames per warp, one and three captures
    for tail in (4, 8, 12):
        L = 2 * (512 * 20 + 1024) + tail
        for n, fpw in ((1, 1), (3, 3), (1, 3)):
            iq = _synth_bytes(n * L, tail + n)
            run("spectrum", [iq, hann], [(1024 * n, np.float32)],
                lambda i, o: [i[0], n, L, i[1], fpw, 0, 0.0, o[0]])
            run("spectrum", [iq, hann], [(1024 * n, np.float32)],
                lambda i, o: [i[0], n, L, i[1], fpw, 1, 0.1, o[0]])

    # FP32 WBFM and AM: a ragged chunk and a ragged last tile (51 200 bytes per tile), several segments, a last
    # segment of one tile (tps 1 and 3 over four tiles), several captures
    L = 51_200 * 3 + 400 * 5 + 48
    for n, tps in ((2, 1), (2, 3), (1, 0)):
        iq = _synth_bytes(n * L, 10 + tps)
        m1 = -(-(L // 2) // 10)
        m2 = -(-m1 // 5)
        run("wbfm_batch", [iq], [(m2 * n, np.float32), (m1 * n, np.float32)], lambda i, o: [i[0], n, L, tps, o[0], o[1]])
        run("wbfm_batch", [iq], [(m2 * n, np.float32)], lambda i, o: [i[0], n, L, tps, o[0], None])
        q = -(-(L // 2) // 20)
        q = -(-q // 10)
        m3 = -(-2 * q // 3)
        run("am_batch", [iq], [(m3 * n, np.float32), (q * n, np.float32)], lambda i, o: [i[0], n, L, tps, o[0], o[1]])

    # tensor-core engine: a ragged last row (320 bytes per row, 40 000 bytes per tile) and several segments
    L = 40_000 * 2 + 320 * 3 + 48
    for n, tps in ((2, 1), (1, 2), (3, 0)):
        iq = _synth_bytes(n * L, 20 + tps)
        m1 = -(-(L // 2) // 10)
        m2 = -(-m1 // 5)
        run("wbfm_tc_batch", [iq], [(m2 * n, np.float32), (m1 * n, np.float32)],
            lambda i, o: [i[0], n, L, tps, o[0], o[1], None, None])

    # streaming steps with carried state: every launch gets exactly its chunks
    plain = run.plain
    ch = plain.emu_fm_chunk()
    for tps in (0, 1):
        iq = _synth_bytes(2 * ch * 400, 30 + tps)
        fm_state = [np.zeros(plain.emu_sizeof_fm_state(), np.uint8) for _ in range(2)]
        am_f = [np.zeros(plain.emu_sizeof_am_front_state(), np.uint8) for _ in range(2)]
        am_b = [np.zeros(plain.emu_sizeof_am_back_state(), np.uint8) for _ in range(2)]
        pos = 0
        for k in (1, 2, 130, 3, 264):
            blk = iq[2 * ch * pos:2 * ch * (pos + k)]
            a0, a1 = -(-pos * (ch // 10) // 5), -(-(pos + k) * (ch // 10) // 5)
            for lib, state, prep in ((run.asan, fm_state[0], _exact), (plain, fm_state[1], _padded)):
                x = prep(blk)
                a, d, na = np.full(a1 - a0, np.nan, np.float32), np.full(k * (ch // 10), np.nan, np.float32), C.c_uint32()
                lib.emu_wbfm_stream(x.ctypes.data, k, pos, state.ctypes.data, a.ctypes.data, C.byref(na), d.ctypes.data, tps)
                assert na.value == a.size
                if lib is plain:
                    assert a.tobytes() == a_asan.tobytes() and d.tobytes() == d_asan.tobytes(), "wbfm_stream"
                a_asan, d_asan = a, d
            b0, b1 = (2 * pos + 2) // 3, (2 * (pos + k) + 2) // 3
            for lib, fs, bs, prep in ((run.asan, am_f[0], am_b[0], _exact), (plain, am_f[1], am_b[1], _padded)):
                x = prep(blk)
                a, na = np.full(b1 - b0, np.nan, np.float32), C.c_uint32()
                lib.emu_am_stream(x.ctypes.data, k, pos, fs.ctypes.data, bs.ctypes.data, a.ctypes.data, C.byref(na), tps)
                assert na.value == a.size
                if lib is plain:
                    assert a.tobytes() == am_asan.tobytes(), "am_stream"
                am_asan = a
            assert fm_state[0].tobytes() == fm_state[1].tobytes() and am_f[0].tobytes() == am_f[1].tobytes()
            pos += k
            run.count += 2

    # counter check from odd word offsets: the buffer ends exactly where the block ends
    for nbytes, off in ((4, 4), (20, 12), (2048 + 36, 4), (16384 + 2048 + 20, 12)):
        raw = np.empty(off + nbytes, np.uint8)
        raw[off:] = (np.arange(nbytes) + 250) % 256
        raw[off + nbytes // 2] ^= 0x10
        res = []
        for lib, buf in ((run.asan, raw), (plain, _padded(raw))):
            n, f = C.c_uint64(), C.c_uint64()
            lib.emu_counter_check(buf.ctypes.data + off, nbytes, 250, C.byref(n), C.byref(f), None, 0)
            res.append((n.value, f.value))
        assert res[0] == res[1], ("counter_check", nbytes, off)
        run.count += 1

    # conversion, generator, render
    for nbytes in (16, 2064, 16 * 1500):
        iq = _synth_bytes(nbytes, nbytes)
        run("convert_cf32", [iq], [(nbytes, np.float32)], lambda i, o: [i[0], nbytes, None, o[0]])
        run("convert_cf32", [iq, hann], [(nbytes, np.float32)], lambda i, o: [i[0], nbytes, i[1], o[0]])
    lut = np.sin(2 * np.pi * (np.arange(4097) % 4096) / 4096).astype(np.float32)
    for kind in range(4):
        run("synth", [lut], [(3 * 4816, np.uint8)], lambda i, o: [o[0], 3, 4816, kind, 5, i[0]])
    rng = np.random.default_rng(1)
    for rows in (1, 3, 100):
        spectra = (np.abs(rng.standard_normal((rows, 1024))) * 10.0 ** rng.uniform(0, 9, (rows, 1024))).astype(np.float32)
        run("render_spectrum", [spectra], [(rows * 272 * 480, np.uint32)], lambda i, o: [i[0], rows, 1.0, 0.0, 100.0, o[0]])
        run("render_waterfall", [spectra], [(272 * 480, np.uint32)], lambda i, o: [i[0], rows, 1.0, 0.0, 100.0, o[0]])
    print(f"checked {run.count} calls")


if __name__ == "__main__":
    _child(sys.argv[1], sys.argv[2])
