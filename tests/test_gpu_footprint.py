"""Where every kernel writes and reads: exactly its outputs, only its inputs.

The value tests read outputs from buffers whose old contents may already be the right answer (a host array from
np.empty, batch_host's result staging kept in the context, a fresh cudaMalloc that returns the block the previous
identical call just freed), so an element a kernel never writes can pass them, and a write past the end of an output
or a read past the end of a capture goes unseen.  Here every output lies inside a guard band of G bytes on each side,
and each call runs twice: once with everything filled with sentinel A, once with sentinel B (two NaN bit patterns no
kernel produces; 0x00 and 0xFF for byte outputs).  Then
  1. both guards still hold their fill: nothing was written outside the output;
  2. the two payloads are bitwise identical: every element was written, and none depends on the old contents;
  3. the payload is finite and matches the float64 golden model within the tolerances of test_gpu_parity.py.
Inputs lie inside guard bands too.  The same call with random bytes instead of zeros around the captures, and
inside a batch with other bytes in the neighbouring captures, must give bitwise the same outputs for the capture
that did not change: the batch shape, hence the launch plan, is the same.

G = 1 MiB is larger than any tile's input or output span, so a plausible overrun stays inside the allocation.
The shapes come from test_gpu_plan_regimes.py, which pins each one to its launch-plan regime.
"""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle_api import AVG_EMA, AVG_MEAN, SYNTH_AM, SYNTH_COUNTER, SYNTH_MULTITONE, SYNTH_WBFM, WIN_BLACKMAN, WIN_HANN, \
    WIN_RECT, Golden, wrap_phase
from test_gpu_parity import AM_AUDIO_ATOL, DISC_ATOL, FM_AUDIO_ATOL, spec_check, spec_check_few_frames
from test_gpu_plan_regimes import FP32_SHAPES, SPEC_FPW, TC_SHAPES, UNALIGNED, assert_regime
from test_render import gold_render, gold_waterfall

pytestmark = pytest.mark.gpu

G = 1 << 20
SENTINELS = (0x7FA5A5A5, 0xFFC3C3C3)  # NaN bit patterns for float and word outputs
BYTE_SENTINELS = (0x00, 0xFF)         # for byte outputs
WAVE_LEN = (64 << 20) + 16            # three captures of this length run as waves of two and one (test_gpu_plan_regimes)


# ------------------------------------------------------------------------------------------ harness
def fill_bytes(nbytes, sentinel, byte_sentinel):
    if byte_sentinel:
        return np.full(nbytes, sentinel, np.uint8)
    return np.full(-(-nbytes // 4), sentinel, np.uint32).view(np.uint8)[:nbytes]


def assert_guards(raw, fill, start, n, what):
    """raw / fill: the whole guarded region as bytes; the payload is raw[start:start + n]"""
    for name, sl in (("before", slice(0, start)), ("after", slice(start + n, raw.size))):
        bad = np.flatnonzero(raw[sl] != fill[sl])
        if bad.size:
            at = bad + sl.start - start
            raise AssertionError(f"{what}: {bad.size} bytes written {name} the payload, at payload offsets "
                                 f"{at.min()} .. {at.max()} (payload {n} bytes)")


class DevRegion:
    """G + offset + n + G bytes of device memory; the payload starts `offset` bytes after a 256-byte boundary"""

    def __init__(self, s, n, offset=0):
        self.s, self.n, self.offset = s, n, offset
        self.total = 2 * G + offset + n
        self.base = s.dev_alloc(self.total)
        self.ptr = self.base + G + offset

    def put(self, payload, guard_rng=None):
        """payload bytes, with zeros (guard_rng None) or seeded random bytes around them"""
        head, tail = G + self.offset, G
        for ptr, k in ((self.base, head), (self.ptr + self.n, tail)):
            self.s.to_dev(ptr, np.zeros(k, np.uint8) if guard_rng is None else guard_rng.integers(0, 256, k, dtype=np.uint8))
        self.s.to_dev(self.ptr, payload)

    def free(self):
        self.s.dev_free(self.base)


def footprint(s, inputs, out_bytes, launch, byte_out=False, variants=(), seed=0):
    """Run `launch(in_ptrs, out_ptrs)` on guarded device buffers:
      - with sentinel A and with sentinel B in the outputs, zeros around the inputs;
      - with sentinel A, seeded random bytes around the inputs;
      - with sentinel A for every variant (a list of replacement inputs; the caller compares what must not change).
    Asserts that no run writes outside its outputs, that the first three give bitwise the same outputs, and that
    float outputs are finite.  inputs: [(uint8 array, byte offset)].  Returns (outputs, [outputs of each variant]) as
    uint8 arrays."""
    ins = [DevRegion(s, a.size, off) for a, off in inputs]
    outs = [DevRegion(s, n) for n in out_bytes]
    sents = BYTE_SENTINELS if byte_out else SENTINELS
    try:
        def run(sentinel, arrays, guard_rng):
            for r, a in zip(ins, arrays):
                r.put(a, guard_rng)
            fills = [fill_bytes(r.total, sentinel, byte_out) for r in outs]
            for r, f in zip(outs, fills):
                s.to_dev(r.base, f)
            launch([r.ptr for r in ins], [r.ptr for r in outs])
            s.sync()
            got = []
            for i, (r, f) in enumerate(zip(outs, fills)):
                raw = s.to_host(r.base, r.total)
                assert_guards(raw, f, G, r.n, f"output {i} (sentinel {sentinel:#x})")
                got.append(raw[G:G + r.n].copy())
            return got

        base = [a for a, _ in inputs]
        first = run(sents[0], base, None)
        for sentinel, rng in ((sents[1], None), (sents[0], np.random.default_rng(seed))):
            again = run(sentinel, base, rng)
            for i, (a, b) in enumerate(zip(first, again)):
                assert np.array_equal(a, b), (f"output {i} differs between runs (sentinel {sentinel:#x}, "
                                              f"{'random' if rng else 'zero'} input guards) at "
                                              f"{np.flatnonzero(a != b)[:8].tolist()} ...")
        if not byte_out:
            for i, a in enumerate(first):
                bad = np.flatnonzero(~np.isfinite(a.view(np.float32)))
                assert not bad.size, f"output {i}: {bad.size} elements not finite, first at {bad[:8].tolist()}"
        rng = np.random.default_rng(seed + 1)
        var = [run(sents[0], v, rng) for v in variants]
        return first, var
    finally:
        for r in ins + outs:
            r.free()


def as_f32(b, rows=1):
    return b.view(np.float32).reshape(rows, -1)


def keep_only(iq, len_each, keep):
    """the batch with every capture but `keep` replaced by other bytes"""
    v = ~iq
    v[keep * len_each:(keep + 1) * len_each] = iq[keep * len_each:(keep + 1) * len_each]
    return v


def neighbour_variants(iq, n_captures, len_each):
    """capture 0 and the last capture, each with different neighbours"""
    if n_captures < 2:
        return [], []
    keeps = [0, n_captures - 1]
    return keeps, [[keep_only(iq, len_each, k)] for k in keeps]


def picks(n_captures, seed):
    """the captures checked against the golden model: the first, the last and one seeded pick"""
    return sorted({0, n_captures - 1, int(np.random.default_rng(seed).integers(0, n_captures))})


# -------------------------------------------------------------------------------- golden, cached
@functools.lru_cache(maxsize=None)
def golden():
    return Golden()


@functools.lru_cache(maxsize=4)
def synth(n_captures, len_each, kind, seed):
    a = golden().synth(n_captures, len_each, kind, seed)
    a.flags.writeable = False
    return a


@functools.lru_cache(maxsize=None)
def gold_spectrum(n_captures, len_each, seed, c, avg_mode):
    iq = synth(n_captures, len_each, SYNTH_MULTITONE, seed)
    return golden().spectrum(iq[c * len_each:(c + 1) * len_each], avg_mode=avg_mode, beta=0.1)[0]


@functools.lru_cache(maxsize=None)
def gold_wbfm(n_captures, len_each, seed, c):
    iq = synth(n_captures, len_each, SYNTH_WBFM, seed)
    return golden().wbfm(iq[c * len_each:(c + 1) * len_each], want_disc=True)


@functools.lru_cache(maxsize=None)
def gold_am(n_captures, len_each, seed, c):
    iq = synth(n_captures, len_each, SYNTH_AM, seed)
    return golden().am(iq[c * len_each:(c + 1) * len_each])


# ------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def ctxs(sdr_lib):
    made = {}

    def get(key):
        if key not in made:
            kw = {"fp32": {}, "tensor": {"fir_engine": sdr_lib.FIR_ENGINE_TENSOR},
                  "mean": {"chains": sdr_lib.CHAIN_SPECTRUM},
                  "ema": {"chains": sdr_lib.CHAIN_SPECTRUM, "avg_mode": AVG_EMA, "ema_beta": 0.1}}[key]
            made[key] = sdr_lib.B200Sdr(**kw)
        return made[key]
    yield get
    for s in made.values():
        s.close()


# ------------------------------------------------------------------------------------------ spectrum
SPECTRUM_CASES = ([pytest.param(1, L, 0, avg, f"spectrum_fpw{fpw}", id=f"fpw{fpw}-{'mean' if avg == AVG_MEAN else 'ema'}")
                   for fpw, (L, _) in sorted(SPEC_FPW.items()) for avg in (AVG_MEAN, AVG_EMA)]
                  + [pytest.param(n, L, 2, AVG_MEAN, f"spectrum_unaligned_{n}", id=f"unaligned{n}x{L}-offset2")
                     for n, L in UNALIGNED]
                  + [pytest.param(1, 262_144, 0, AVG_MEAN, None, id="folded_finalize_256KiB"),
                     pytest.param(3, 2044, 0, AVG_MEAN, None, id="no_frame_memset")])


@pytest.mark.parametrize("n,L,offset,avg,regime", SPECTRUM_CASES)
def test_spectrum_footprint(ctxs, sms, n, L, offset, avg, regime):
    if regime:
        assert_regime(regime, sms)
    s = ctxs("mean" if avg == AVG_MEAN else "ema")
    seed = 300 + n
    iq = synth(n, L, SYNTH_MULTITONE, seed)
    keeps, variants = neighbour_variants(iq, n, L)
    (out,), var = footprint(s, [(iq, offset)], [4096 * n], lambda i, o: s.batch_spectrum_dev(i[0], n, L, o[0]),
                            variants=variants, seed=seed)
    out = as_f32(out, n)
    for k, (v,) in zip(keeps, var):
        assert np.array_equal(as_f32(v, n)[k], out[k]), f"capture {k} changed with its neighbours"
    for c in range(n):
        gold = gold_spectrum(n, L, seed, c, avg)
        if not gold.any():  # shorter than one frame: the spectrum is defined as zeros
            assert not out[c].any()
        elif avg == AVG_MEAN:
            spec_check(out[c], gold)
        else:
            spec_check_few_frames(out[c], gold)


# ------------------------------------------------------------------------------------------ WBFM
WBFM_SHAPES = ([(L, n, f"fp32_{L}x{n}") for L, n in FP32_SHAPES] + [(L, n, f"tc_{L}x{n}") for L, n in TC_SHAPES]
               + [(16, 1, None), (320, 1, None), (2416, 1, None), (4096, 300, None)])


@pytest.mark.parametrize("engine", ["fp32", "tensor"])
@pytest.mark.parametrize("L,n,regime", WBFM_SHAPES, ids=[f"{n}x{L}" for L, n, _ in WBFM_SHAPES])
def test_wbfm_footprint(sdr_lib, ctxs, sms, engine, L, n, regime):
    if regime:
        assert_regime(regime, sms)
    s = ctxs(engine)
    seed = 400 + n
    iq = synth(n, L, SYNTH_WBFM, seed)
    na, nd = sdr_lib.wbfm_audio_len(L), sdr_lib.wbfm_disc_len(L)
    keeps, variants = neighbour_variants(iq, n, L)
    (audio, disc), var = footprint(s, [(iq, 0)], [4 * na * n, 4 * nd * n],
                                   lambda i, o: s.batch_wbfm_dev(i[0], n, L, o[0], o[1]), variants=variants, seed=seed)
    # without the discriminator output: the same audio, bit for bit
    (audio_only,), _ = footprint(s, [(iq, 0)], [4 * na * n], lambda i, o: s.batch_wbfm_dev(i[0], n, L, o[0], None),
                                 seed=seed)
    assert np.array_equal(audio_only, audio)
    audio, disc = as_f32(audio, n), as_f32(disc, n)
    for k, (va, vd) in zip(keeps, var):
        assert np.array_equal(as_f32(va, n)[k], audio[k]) and np.array_equal(as_f32(vd, n)[k], disc[k]), \
            f"capture {k} changed with its neighbours"
    for c in picks(n, seed):
        ga, gd = gold_wbfm(n, L, seed, c)
        assert np.max(np.abs(wrap_phase(disc[c] - gd))) <= DISC_ATOL
        assert np.max(np.abs(audio[c] - ga)) <= FM_AUDIO_ATOL


@pytest.mark.parametrize("L", [16, 2416, 39_856])
def test_tensor_engine_reads_nothing_past_a_ragged_capture(sdr_lib, ctxs, L):
    """A capture of less than one tile with a ragged last row: its only tile is filled by the bounds-checked cp.async
    path.  The raw accumulators of that tile hold the outputs past the capture's end too, which the audio and
    discriminator never show: with zeros or random bytes after the capture they must be bitwise the same, and equal
    to the integer FIR of the capture with u[n] = 0 outside it."""
    s = ctxs("tensor")
    iq = synth(1, L, SYNTH_WBFM, 450)
    runs = []
    for sentinel, guard_rng in ((SENTINELS[0], None), (SENTINELS[1], None), (SENTINELS[0], np.random.default_rng(L))):
        d = DevRegion(s, L)
        acc = HostRegion(128 * 112, np.int32, sentinel)
        q = np.zeros((3, 80), np.int8)
        try:
            d.put(iq, guard_rng)
            s._check(s.lib.b200sdr_debug_wbfm_tc_acc(s.ctx, d.ptr, L, acc.view.ctypes.data, q.ctypes.data, None),
                     "b200sdr_debug_wbfm_tc_acc")
        finally:
            d.free()
        acc.check("accumulators")
        runs.append(acc.view.reshape(128, 112).copy())
    for a in runs[1:]:
        assert np.array_equal(a, runs[0]), f"accumulators depend on the bytes after the capture at {np.argwhere(a != runs[0])[:4].tolist()}"
    n = L // 2
    u = iq.reshape(n, 2).astype(np.int64)
    m = 16 * np.arange(125)[:, None] - 1 + np.arange(17)[None, :]   # column 34 s + 2 j + c of row r: output 16 r - 1 + j
    k = 10 * m[..., None] - np.arange(80)                            # sample index of tap t
    x = np.where(((k >= 0) & (k < n))[..., None], u[np.clip(k, 0, n - 1)], 0)
    want = np.einsum("st,rjtc->rsjc", q.astype(np.int64), x).reshape(125, 102)
    assert np.array_equal(runs[0][:125, :102], want)


# ------------------------------------------------------------------------------------------ AM
AM_SHAPES = [(L, n, f"fp32_{L}x{n}") for L, n in FP32_SHAPES] + [(16, 1, None), (4816, 1, None)]


@pytest.mark.parametrize("L,n,regime", AM_SHAPES, ids=[f"{n}x{L}" for L, n, _ in AM_SHAPES])
def test_am_footprint(sdr_lib, ctxs, sms, L, n, regime):
    if regime:
        assert_regime(regime, sms)
    s = ctxs("fp32")
    seed = 500 + n
    iq = synth(n, L, SYNTH_AM, seed)
    na = sdr_lib.am_audio_len(L)
    keeps, variants = neighbour_variants(iq, n, L)
    (audio,), var = footprint(s, [(iq, 0)], [4 * na * n], lambda i, o: s.batch_am_dev(i[0], n, L, o[0]),
                              variants=variants, seed=seed)
    audio = as_f32(audio, n)
    for k, (v,) in zip(keeps, var):
        assert np.array_equal(as_f32(v, n)[k], audio[k]), f"capture {k} changed with its neighbours"
    for c in picks(n, seed):
        ga = gold_am(n, L, seed, c)
        assert audio[c].size == ga.size and np.max(np.abs(audio[c] - ga)) <= AM_AUDIO_ATOL


# ------------------------------------------------------------------------------- conversion, generator
@pytest.mark.parametrize("window", [WIN_RECT, WIN_HANN, WIN_BLACKMAN], ids=["rect", "hann", "blackman"])
@pytest.mark.parametrize("nbytes", [16, 2064, 262_160])
def test_convert_footprint(ctxs, window, nbytes):
    s = ctxs("fp32")
    iq = np.random.default_rng(nbytes).integers(0, 256, nbytes, dtype=np.uint8)
    (out,), _ = footprint(s, [(iq, 0)], [4 * nbytes],
                          lambda i, o: s._check(s.lib.b200sdr_convert_cf32_dev(s.ctx, i[0], nbytes, window, o[0]),
                                                "b200sdr_convert_cf32_dev"), seed=nbytes)
    out = out.view(np.float32)
    g = golden()
    if window == WIN_RECT:
        assert np.array_equal(out.astype(np.float64), g.convert(iq))
    else:  # one rounded fp32 multiply by the fp32 window value (test_gpu_parity.test_convert_windowed)
        w32 = g.window(window).astype(np.float32)
        want = (g.convert(iq).astype(np.float32).reshape(-1, 2) * np.resize(w32, nbytes // 2)[:, None]).reshape(-1)
        assert np.array_equal(out, want)


@pytest.mark.parametrize("kind", [SYNTH_COUNTER, SYNTH_MULTITONE, SYNTH_WBFM, SYNTH_AM])
def test_synth_fill_footprint(ctxs, kind):
    s = ctxs("fp32")
    n, L = 3, 4816
    (out,), _ = footprint(s, [], [n * L], lambda i, o: s.synth_fill_dev(o[0], n, L, kind, first_capture=9), byte_out=True)
    assert np.array_equal(out, golden().synth(n, L, kind, 9))


# ------------------------------------------------------------------------------------------ counter check
class HostRegion:
    """a numpy view of `count` items inside G bytes of guard on each side"""

    def __init__(self, count, dtype, sentinel, byte_sentinel=False, guard=G):
        self.dtype = np.dtype(dtype)
        self.n = count * self.dtype.itemsize
        self.guard = guard
        self.fill = fill_bytes(2 * guard + self.n, sentinel, byte_sentinel)
        self.raw = self.fill.copy()
        self.view = self.raw[guard:guard + self.n].view(self.dtype)

    def check(self, what):
        assert_guards(self.raw, self.fill, self.guard, self.n, what)


@pytest.mark.parametrize("expect_first", [-1, 7])
def test_counter_check_footprint(ctxs, expect_first):
    s = ctxs("fp32")
    n, L = 5, 16_400
    iq = np.array(synth(n, L, SYNTH_COUNTER, 0))
    rng = np.random.default_rng(5)
    for c in (1, 3):
        hits = c * L + rng.integers(0, L, 4)
        iq[hits] = rng.integers(0, 256, hits.size, dtype=np.uint8)
    iq[4 * L + L - 1] ^= 1  # the last byte of the last capture
    want = [golden().counter_check(iq[c * L:(c + 1) * L], expect_first) for c in range(n)]
    results = []
    for sentinel, guard_rng in ((SENTINELS[0], None), (SENTINELS[1], None), (SENTINELS[0], np.random.default_rng(6))):
        d = DevRegion(s, iq.size)
        try:
            d.put(iq, guard_rng)
            nb, fb = HostRegion(n, np.uint64, sentinel), HostRegion(n, np.uint64, sentinel)
            s._check(s.lib.b200sdr_counter_check_dev(s.ctx, d.ptr, n, L, expect_first,
                                                     nb.view.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                     fb.view.ctypes.data_as(C.POINTER(C.c_uint64))), "counter_check_dev")
        finally:
            d.free()
        nb.check("n_breaks")
        fb.check("first_break")
        results.append((nb.view.copy(), fb.view.copy()))
    for nb, fb in results:
        assert np.array_equal(nb, results[0][0]) and np.array_equal(fb, results[0][1])
        got = [(int(a), None if int(b) == 2**64 - 1 else int(b)) for a, b in zip(nb, fb)]
        assert got == want


# ------------------------------------------------------------------------------------------ render
def render_dev(s, name, ptr, count, out):
    fn = getattr(s.lib, name)
    fn.restype = C.c_int32
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_void_p]
    s._check(fn(s.ctx, ptr, count, 1.0, 0.0, 100.0, out), name)


def random_spectra(rows, seed):
    rng = np.random.default_rng(seed)
    return (np.abs(rng.standard_normal((rows, 1024))) * 10.0 ** rng.uniform(0, 9, (rows, 1024))).astype(np.float32)


@pytest.mark.parametrize("n_spectra", [1, 3])
def test_render_spectrum_footprint(ctxs, n_spectra):
    s = ctxs("mean")
    spectra = random_spectra(n_spectra, n_spectra)
    (img,), _ = footprint(s, [(spectra.view(np.uint8).reshape(-1), 0)], [n_spectra * 272 * 480 * 4],
                          lambda i, o: render_dev(s, "b200sdr_render_spectrum_dev", i[0], n_spectra, o[0]), byte_out=True)
    img = img.view(np.uint32).reshape(n_spectra, 272, 480)
    for k in range(n_spectra):
        assert np.array_equal(img[k], gold_render(golden(), spectra[k], 0.0, 100.0))


@pytest.mark.parametrize("n_rows", [100, 300])
def test_render_waterfall_footprint(ctxs, n_rows):
    """fewer rows than the panel's 272 (the kernel must not read past them), and more (it reads the first 272 only)"""
    s = ctxs("mean")
    spectra = random_spectra(n_rows, n_rows)
    variants = []
    if n_rows > 272:
        other = spectra.copy()
        other[272:] = random_spectra(n_rows - 272, 1)
        variants = [[other.view(np.uint8).reshape(-1)]]
    (img,), var = footprint(s, [(spectra.view(np.uint8).reshape(-1), 0)], [272 * 480 * 4],
                            lambda i, o: render_dev(s, "b200sdr_render_waterfall_dev", i[0], n_rows, o[0]),
                            byte_out=True, variants=variants)
    for (v,) in var:
        assert np.array_equal(v, img), "the image depends on rows past the panel's 272"
    assert np.array_equal(img.view(np.uint32).reshape(272, 480), gold_waterfall(golden(), spectra[:272], 0.0, 100.0))


# ------------------------------------------------------------------------------------------ split capture
@pytest.mark.parametrize("with_data", [True, False], ids=["data", "empty_rank"])
def test_split_spectrum_footprint(sdr_lib, with_data):
    L = 262_144 + 4096
    iq = synth(1, L, SYNTH_MULTITONE, 600)
    frames = (L // 2 - 1024) // 512 + 1
    with sdr_lib.B200Sdr(chains=sdr_lib.CHAIN_SPECTRUM) as s:
        s.exchange_create(1, 0)
        s.exchange_connect([b""])

        def launch(i, o):
            s.split_spectrum_dev(i[0], L if with_data else 0, frames, o[0])
            s.exchange_wait()
        (out,), _ = footprint(s, [(iq, 0)], [4096], launch, seed=600)
        s.exchange_destroy()
    out = out.view(np.float32)
    if with_data:
        spec_check(out, gold_spectrum(1, L, 600, 0, AVG_MEAN))
    else:
        assert not out.any()


# ------------------------------------------------------------------------------------------ batch_host
BATCH_HOST_CASES = [pytest.param(1_689_616, 2, id="2x1689616"), pytest.param(WAVE_LEN, 3, id="waves")]


def dev_reference(s, iq, n, L, fm_len, am_len):
    """spectrum, WBFM audio and AM audio of the captures of `iq` through the _dev entry points in one launch each
    (outputs with room behind them: an overrun is the footprint tests' finding, not a fault here)"""
    d_iq = s.dev_alloc(iq.size)
    outs = [s.dev_alloc(4 * k * n + G) for k in (1024, fm_len, am_len)]
    try:
        s.to_dev(d_iq, iq)
        s.batch_spectrum_dev(d_iq, n, L, outs[0])
        s.batch_wbfm_dev(d_iq, n, L, outs[1])
        s.batch_am_dev(d_iq, n, L, outs[2])
        s.sync()
        return [s.to_host(d, 4 * k * n, np.float32).reshape(n, k) for d, k in zip(outs, (1024, fm_len, am_len))]
    finally:
        for d in [d_iq] + outs:
            s.dev_free(d)


@pytest.mark.parametrize("engine", ["fp32", "tensor"])
@pytest.mark.parametrize("L,n", BATCH_HOST_CASES)
def test_batch_host_footprint(sdr_lib, ctxs, sms, engine, L, n):
    """host outputs as views into guarded arrays.  The result staging is kept in the context between calls, so a
    call over other bytes runs between the two sentinel runs: an element the kernels skip then differs."""
    if L == WAVE_LEN:
        assert_regime("waves", sms)
    s = ctxs(engine)
    chains = sdr_lib.CHAIN_SPECTRUM | sdr_lib.CHAIN_WBFM | sdr_lib.CHAIN_AM
    kinds = (SYNTH_MULTITONE, SYNTH_WBFM, SYNTH_AM)
    iq = np.concatenate([golden().synth(1, L, kinds[c % 3], 700 + c) for c in range(n)])
    lens = (1024, sdr_lib.wbfm_audio_len(L), sdr_lib.am_audio_len(L))
    runs = []
    for sentinel in SENTINELS:
        # a copy-back of one capture too many stays inside the guard
        regions = [HostRegion(k * n, np.float32, sentinel, guard=max(G, 4 * k)) for k in lens]
        s.batch_host(chains, iq, n, L, *[r.view for r in regions])
        for r, what in zip(regions, ("spectrum", "wbfm", "am")):
            r.check(what)
        runs.append([r.view.reshape(n, -1).copy() for r in regions])
        if sentinel == SENTINELS[0]:  # other results into the staging buffers
            scratch = [HostRegion(k * n, np.float32, sentinel, guard=max(G, 4 * k)) for k in lens]
            s.batch_host(chains, ~iq, n, L, *[r.view for r in scratch])
    for a, b, what in zip(*runs, ("spectrum", "wbfm", "am")):
        assert np.all(np.isfinite(a)), what
        assert np.array_equal(a, b), f"{what}: differs between runs at {np.argwhere(a != b)[:4].tolist()}"
    per_wave = max(1, min((192 << 20) // L, n))
    for c0 in range(0, n, per_wave):  # each wave against the _dev entry points over the same captures
        nc = min(per_wave, n - c0)
        ref = dev_reference(s, iq[c0 * L:(c0 + nc) * L], nc, L, lens[1], lens[2])
        for got, want, what in zip(runs[0], ref, ("spectrum", "wbfm", "am")):
            assert np.array_equal(got[c0:c0 + nc], want), f"{what}, wave at capture {c0}"


# ------------------------------------------------------------------------------------------ streaming getters
def stream(sdr_lib, iq, block):
    s = sdr_lib.B200Sdr(chains=sdr_lib.CHAIN_SPECTRUM | sdr_lib.CHAIN_WBFM | sdr_lib.CHAIN_AM)
    for a in range(0, iq.size, block):
        s.process_samples(iq[a:a + block])
    return s


def get_audio_raw(s, chain, capacity, sentinel):
    r = HostRegion(capacity, np.float32, sentinel)
    n = C.c_uint32(0xFFFFFFFF)
    s._check(s.lib.b200sdr_get_audio(s.ctx, chain, r.view.ctypes.data, capacity, C.byref(n)), "b200sdr_get_audio")
    r.check(f"get_audio capacity {capacity}")
    assert n.value <= capacity
    tail = r.view[n.value:].view(np.uint32)
    assert np.all(tail == sentinel), f"get_audio wrote past n_out = {n.value}"
    return r.view[:n.value].copy()


@pytest.mark.parametrize("chain", ["wbfm", "am"])
def test_get_audio_footprint(sdr_lib, chain):
    """a capacity below what is queued, then one above what is left: exactly n_out floats written each time"""
    total = 262_144 * 2 + 4000
    iq = synth(1, total, SYNTH_WBFM if chain == "wbfm" else SYNTH_AM, 800)
    bit = sdr_lib.CHAIN_WBFM if chain == "wbfm" else sdr_lib.CHAIN_AM
    queued = sdr_lib.wbfm_stream_audio_len(total) if chain == "wbfm" else (2 * (total // 2 // 200) + 2) // 3
    pops = []
    for sentinel in SENTINELS:
        s = stream(sdr_lib, iq, 131_072)
        try:
            a = get_audio_raw(s, bit, queued - 100, sentinel)
            b = get_audio_raw(s, bit, 150, sentinel)
            assert (a.size, b.size) == (queued - 100, 100)
            assert get_audio_raw(s, bit, 16, sentinel).size == 0
        finally:
            s.close()
        pops.append(np.concatenate([a, b]))
    assert np.array_equal(pops[0], pops[1])
    g = golden()
    if chain == "wbfm":
        assert np.max(np.abs(pops[0] - g.wbfm(iq)[:queued])) <= FM_AUDIO_ATOL
    else:
        assert np.max(np.abs(pops[0] - g.am(iq)[:queued])) <= AM_AUDIO_ATOL


def test_streaming_getters_footprint(sdr_lib):
    """get_spectrum writes 1024 floats, debug_last_block at most its capacity, get_taps nothing when the capacity is
    too small and exactly the taps otherwise"""
    total = 262_144 + 4000
    iq = synth(1, total, SYNTH_MULTITONE, 900)
    s = stream(sdr_lib, iq, 262_144)
    try:
        specs = []
        for sentinel in SENTINELS:
            r = HostRegion(1024, np.float32, sentinel)
            frames = C.c_uint64(0)
            s._check(s.lib.b200sdr_get_spectrum(s.ctx, r.view.ctypes.data, C.byref(frames)), "b200sdr_get_spectrum")
            r.check("get_spectrum")
            specs.append(r.view.copy())
        assert np.array_equal(specs[0], specs[1])
        spec_check(specs[0], golden().spectrum(iq)[0])

        for sentinel in BYTE_SENTINELS:
            r = HostRegion(100, np.uint8, sentinel, byte_sentinel=True)
            n = C.c_uint32(0)
            s._check(s.lib.b200sdr_debug_last_block(s.ctx, r.view.ctypes.data, 100, C.byref(n)), "b200sdr_debug_last_block")
            r.check("debug_last_block")
            assert n.value == 4000 and np.array_equal(r.view, iq[262_144:262_144 + 100])

        g = golden()
        for which in range(5):
            want = g.taps(which).astype(np.float32)
            for capacity in (want.size - 1, want.size):
                r = HostRegion(capacity, np.float32, SENTINELS[0])
                n = C.c_uint32(0)
                rc = s.lib.b200sdr_get_taps(s.ctx, which, r.view.ctypes.data, capacity, C.byref(n))
                r.check(f"get_taps({which}, capacity {capacity})")
                assert n.value == want.size
                if capacity < want.size:
                    assert rc == sdr_lib.NOT_SUPPORTED and np.all(r.view.view(np.uint32) == SENTINELS[0])
                else:
                    assert rc == sdr_lib.OK and np.array_equal(r.view, want)
    finally:
        s.close()
