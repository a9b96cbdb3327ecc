"""Pins the oracle: the numpy port (oracle/port.py) against (i) the UNMODIFIED reference (oracle/_ref; its outputs for
these inputs are stored, tests/reference_outputs.py), (ii) the committed golden vectors that library produced
(tests/golden/reference_vectors.npz) and (iii) the reference's own known-answer module tests. CPU only."""
import os

import numpy as np
import pytest

from oracle import port

GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "reference_vectors.npz")


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLDEN)


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


# ---- (ii) golden vectors -------------------------------------------------------------------------

def test_golden_window_bit_exact(gold):
    for n in (8, 4096):
        assert np.array_equal(port.window(n), gold[f"window{n}"])


def test_golden_fft(gold):
    assert rel(port.fft(gold["fft1024_in"]), gold["fft1024_out"]) < 1e-6
    assert abs(abs(gold["fft1024_out"][5]) - 1024.0) < 1e-2          # BASELINE.md §2 sanity value
    assert rel(port.fft(gold["fft256_in"]), gold["fft256_fwd"]) < 1e-6
    assert rel(port.fft(gold["fft256_in"], forward=False), gold["fft256_inv"]) < 1e-6


def test_golden_amplitude_bit_exact_and_range(gold):
    assert np.array_equal(port.amplitude(gold["amp_in"], 512), gold["amp_out"])
    assert np.abs(port.range_(gold["amp_out"], -80.0, -20.0) - gold["range_out"]).max() <= 2.4e-7   # tanhf ulp


def test_golden_chain(gold):
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from parity import assert_db_close, true_spectrum
    x = gold["chain_in"]
    spec = true_spectrum(x, port.invert(port.window(4096)))
    assert_db_close(port.spectrum_engine(x, False), gold["chain_db"], spec)
    assert_db_close(port.spectrum_engine(x, True), gold["chain_scaled"], spec, scale=2.0 / 120.0, floor=3e-7)
    assert int(gold["chain_db"][0].argmax()) == 2048          # row 0: tones at bins 0, 511, 2048 shifted by N/2


def test_golden_filter_taps_bit_exact(gold):
    assert np.array_equal(port.filter_taps(8e6, 1e6, [0.0, 1.5e6], 33), gold["taps33"])


@pytest.mark.parametrize("taps,decim", [(129, 8), (127, 1)])
def test_golden_filter_block(gold, taps, decim):
    block = port.FilterBlock(8e6, 1e6, taps, 1024)
    assert block.R == decim
    for i in range(2):
        got = block(gold[f"filter{taps}_in{i}"])
        want = gold[f"filter{taps}_out{i}"]
        assert got.shape == want.shape
        assert rel(got, want) < 2e-6


def test_filter_chain_equals_time_domain_decimated_convolution(gold):
    """The identity the CUDA kernel relies on (SURVEY.md Appendix B): fold + ifft + 1/M + unpad + overlap-add
    == causal streaming convolution kept at every R-th sample."""
    taps, r = 129, 8
    x = np.concatenate([gold["filter129_in0"].reshape(-1), gold["filter129_in1"].reshape(-1)]).astype(np.complex128)
    h = port.filter_taps(8e6, 1e6, [0.0], taps)[0].astype(np.complex128)
    y = np.convolve(x, h)[: x.size][::r]
    want = np.concatenate([gold["filter129_out0"].reshape(-1), gold["filter129_out1"].reshape(-1)])
    assert rel(y, want) < 2e-6


@pytest.mark.parametrize("de", ["none", "75us"])
def test_golden_fm(gold, de):
    fm = port.FmNarrow(250e3, de, lanes=1)
    for i in range(2):
        x = gold[f"fm_{de}_in{i}"]
        got = fm(x[:, None, :])[:, 0, :]
        want = gold[f"fm_{de}_out{i}"]
        assert np.abs(got - want).max() <= 1e-6                 # atan2f: numpy vs glibc, <= 1-2 ulp


# ---- (i) the compiled reference, when present ------------------------------------------------------

def test_port_matches_compiled_reference(ref):
    from cyberether_b200.synthetic import gaussian_cf32, spectral_rows
    x = gaussian_cf32((5, 1024), 3)
    assert ref.window(1024).equals(port.window(1024))
    w = port.invert(port.window(1024)).reshape(1, 1024)
    assert ref.multiply(x, w).equals(port.multiply(x, w))
    want = ref.fft(x)
    assert np.abs(want.diff(port.fft(x))).max() / want.absmax() < 1e-6
    spectrum = port.fft(x)
    assert ref.amplitude(spectrum).equals(port.amplitude(spectrum, 1024))
    xs = spectral_rows(11, 3)
    assert np.abs(ref.spectrum_engine(xs, True).diff(port.spectrum_engine(xs, True))).max() < 2e-4


# ---- (iii) the reference's own known-answer tests (SURVEY.md §4) --------------------------------------

def test_known_answer_fft_dc_and_roundtrip():
    """src/domains/dsp/fft/module_tests.cc:52-143."""
    out = port.fft(np.ones(64, np.complex64))
    assert abs(out[0].real - 64) < 1e-3 and np.abs(out[1:]).max() < 1e-3
    t = np.arange(64) / 64.0
    x = (np.cos(2 * np.pi * 4 * t) + 1j * np.sin(2 * np.pi * 4 * t)).astype(np.complex64)
    back = port.fft(port.fft(x), forward=False)
    assert np.abs(back / 64 - x).max() < 1e-2


def test_known_answer_amplitude_and_range():
    """amplitude/module_tests.cc (0.1-0.5 dB vs exact log10, -inf at 0); range/module_tests.cc:62-65 (1e-6)."""
    x = np.array([1 + 0j, 0.5 + 0j, 0j, 3 + 4j], np.complex64)
    out = port.amplitude(x, 4)
    exact = 20 * np.log10(np.array([1, 0.5, 1, 5.0])) + 20 * np.log10(1 / 4)
    assert np.isneginf(out[2])
    assert np.abs(out[[0, 1, 3]] - exact[[0, 1, 3]]).max() < 0.1
    r = port.range_(np.array([-1.0, 0.0, 1.0], np.float32), -1.0, 1.0)
    assert np.abs(r - (0.5 + 0.5 * np.tanh(4 * (np.array([0, 0.5, 1.0]) - 0.5)))).max() < 1e-6


@pytest.mark.parametrize("name,np_type,is_complex", [("I8", np.int8, False), ("U16", np.uint16, False),
                                                     ("I32", np.int32, False), ("CI8", np.int8, True),
                                                     ("CU8", np.uint8, True), ("CI16", np.int16, True),
                                                     ("CU32", np.uint32, True)])
def test_port_cast_matches_reference(ref, name, np_type, is_complex):
    info = np.iinfo(np_type)
    shape = (7, 33, 2) if is_complex else (7, 33)
    x = np.random.default_rng(3).integers(info.min, info.max, size=shape, endpoint=True, dtype=np_type)
    want = ref.run_block("cast", {"buffer": x}, {"outputType": "CF32" if is_complex else "F32"}, "buffer",
                         dtypes={"buffer": name})
    assert want.equals(port.cast(x, complex_pairs=is_complex))


@pytest.mark.parametrize("complex_input", [True, False])
@pytest.mark.parametrize("shape,tile", [((3, 1000), 256), ((2, 4096), 4096), ((1, 77), 1024), ((4, 513), 64)])
def test_port_agc_matches_reference(ref, complex_input, shape, tile):
    rng = np.random.default_rng(sum(shape) + tile)
    env = np.exp(rng.uniform(-6, 6, size=(shape[0], 1))) * (1 + 5 * (np.arange(shape[1]) > shape[1] // 2))
    x = rng.standard_normal(shape) * env
    if complex_input:
        x = (x + 1j * rng.standard_normal(shape) * env).astype(np.complex64)
    else:
        x = x.astype(np.float32)
    want = ref.run_block("agc", {"signal": x}, {"tileSize": tile}, "signal")
    # the agc BLOCK holds its parameters as F32 (include/jetstream/domains/dsp/agc/block.hh:9-14) and widens them
    # into the module's F64 config (block_impl.cc:17-24): minGain is (double)0.01f, epsilon (double)1e-12f
    f32 = lambda v: float(np.float32(v))
    got = port.agc(x, tile_size=tile, reference=f32(1.0), epsilon=f32(1e-12), min_gain=f32(0.01), max_gain=f32(100.0),
                   max_gain_change=f32(4.0))
    assert got.dtype == want.dtype
    assert want.equals(got)


# ---- golden vectors of the widened path (cast, agc, SDR-style integer chain) ---------------------------------------

@pytest.mark.parametrize("name", ["I8", "U8", "I16", "U16", "I32", "U32", "CI8", "CU8", "CI16", "CU16", "CI32", "CU32"])
def test_golden_cast_bit_exact(gold, name):
    got = port.cast(gold[f"cast_{name}_in"], complex_pairs=name.startswith("C"))
    assert np.array_equal(got, gold[f"cast_{name}_out"])


@pytest.mark.parametrize("kind", ["f32", "cf32"])
@pytest.mark.parametrize("tile", [128, 700])
def test_golden_agc_bit_exact(gold, kind, tile):
    f32 = lambda v: float(np.float32(v))           # the agc BLOCK widens F32 parameters (block.hh:9-14)
    got = port.agc(gold[f"agc_{kind}_in"], tile_size=tile, reference=f32(1.0), epsilon=f32(1e-12), min_gain=f32(0.01),
                   max_gain=f32(100.0), max_gain_change=f32(4.0))
    assert np.array_equal(got, gold[f"agc_{kind}_tile{tile}"])


@pytest.mark.parametrize("name", ["CI8", "CI16"])
def test_golden_sdr_chain(gold, name):
    """cast -> spectrum_engine on integer captures: the port (cast restatement + chain restatement) against the
    reference flowgraph's output, same bound as the CF32 chain golden."""
    x = port.cast(gold[f"sdr_{name}_in"], complex_pairs=True)
    got = port.spectrum_engine(x, enable_scale=True)
    assert np.abs(got - gold[f"sdr_{name}_agc0"]).max() <= 2e-3


@pytest.mark.parametrize("deemphasis", ["none", "50us"])
def test_port_fm_wide_matches_reference(ref, deemphasis):
    """Wideband (stereo) decoder restatement vs the reference fm module over two cycles with carried state and a NaN
    sample: numpy's F32 cos / sin / atan2 differ from glibc's by an ulp, the recursive filters keep that below 2e-5."""
    rate = 250e3
    rng = np.random.Generator(np.random.PCG64(4))
    cycles = []
    for c in range(2):
        t = (np.arange(2 * 768) + c * 2 * 768) / rate
        left, right = np.sin(2 * np.pi * 1e3 * t), 0.5 * np.sin(2 * np.pi * 3e3 * t)
        mpx = 0.45 * (left + right) + 0.1 * np.sin(2 * np.pi * 19e3 * t) + \
            0.45 * (left - right) * np.sin(2 * np.pi * 38e3 * t)
        phase = 2 * np.pi * 75e3 * np.cumsum(mpx) / rate
        x = np.exp(1j * phase) + 0.002 * (rng.standard_normal(t.size) + 1j * rng.standard_normal(t.size))
        cycles.append(x.astype(np.complex64).reshape(2, 768))
    cycles[1][1, 5] = np.nan + 0j
    decoder = port.FmWide(rate, deemphasis, lanes=1)
    with ref.Session() as s:
        s.add_source("src", cycles[0], 1, 0, -1)                     # sampleAxis 1, batchAxis 0
        s.add_block("fm", "fm", {"mode": "wide", "deemphasis": deemphasis, "sampleRate": rate}, {"signal": "src.signal"})
        for x in cycles:
            s.write_source("src", x)
            s.compute()
            want = s.output("fm", "signal")
            got = decoder(x[:, None, :])[:, 0]
            assert got.shape == want.shape == (2, 768, 2)
            assert want.same_nan(got)
            got, want = want.take(got), want.values
            m = ~np.isnan(want)
            assert np.abs(got[m] - want[m]).max() <= 2e-5


# ---- SURVEY.md §8 f1: lineplot / waterfall consumers — port.py pinned to the reference's own compute TUs ----------------

def test_lineplot_port_matches_reference_module_and_known_answers(ref):
    """Known answers of src/domains/visualization/lineplot/module_tests.cc: -inf input stays finite after the clamp
    (:363-425), a later finite frame raises the average, 2.0 saturates at <= 1; decimation indexes with the ORIGINAL
    row width (:438-457: sums 11 and 33)."""
    from oracle import port
    with ref.VizSession("lineplot", (2, 4), {"averaging": 2}, sample_axis=1, batch_axis=0) as v:
        p = port.Lineplot(4, batches=2, averaging=2)
        v.compute(np.full((2, 4), -np.inf, np.float32))
        first = v.read().array().reshape(-1, 2)
        assert np.all(np.isfinite(first)) and np.array_equal(first, p.compute(np.full((2, 4), -np.inf, np.float32)))
        assert np.array_equal(first[:, 1], np.full(4, -0.5, np.float32))          # clamp(-inf) = -1, EMA over 2
        v.compute(np.ones((2, 4), np.float32))
        second = v.read().array().reshape(-1, 2)
        assert np.array_equal(second, p.compute(np.ones((2, 4), np.float32))) and np.all(second[:, 1] > first[:, 1])
        v.compute(np.full((2, 4), 2.0, np.float32))
        third = v.read().array().reshape(-1, 2)
        assert np.array_equal(third, p.compute(np.full((2, 4), 2.0, np.float32))) and np.all(third[:, 1] <= 1.0)
    x = np.array([[1, 2, 3, 4, 5], [10, 20, 30, 40, 50]], np.float32)
    with ref.VizSession("lineplot", (2, 5), {"decimation": 2}, sample_axis=1, batch_axis=0) as v:
        v.compute(x)
        got = v.read().array().reshape(-1, 2)
    # sums 11, 33 -> amplitude = clamp(sum * (1 / (0.5 * 2)) - 1, -1, 1) = 1, 1
    assert np.array_equal(got[:, 1], np.array([1.0, 1.0], np.float32))
    assert np.array_equal(got, port.Lineplot(5, batches=2, decimation=2).compute(x))


@pytest.mark.parametrize("shape,dec,avg", [((64, 4096), 1, 1), ((64, 4096), 4, 8), ((7, 1000), 3, 2), ((1, 256), 1, 4)])
def test_lineplot_port_random_cycles(ref, shape, dec, avg):
    from oracle import port
    rng = np.random.default_rng(1)
    p = port.Lineplot(shape[1], batches=shape[0], decimation=dec, averaging=avg)
    with ref.VizSession("lineplot", shape, {"decimation": dec, "averaging": avg}, sample_axis=1, batch_axis=0) as v:
        for _ in range(4):
            x = rng.uniform(0.0, 1.2, shape).astype(np.float32)
            v.compute(x)
            assert v.read(select=lambda a: a.reshape(-1, 2)).equals(p.compute(x))


def test_lineplot_sample_and_channel_layouts_are_equivalent(ref):
    """lineplot/module_tests.cc:459-518: [2, 4] batch-leading == [4, 2] batch-trailing, sample or channel axis."""
    lead = np.array([[0.1, 0.2, 0.3, 0.4], [0.2, 0.2, 0.2, 0.2]], np.float32)
    outs = []
    for use_channel in (False, True):
        kw = {"channel_axis": 1} if use_channel else {"sample_axis": 1}
        with ref.VizSession("lineplot", (2, 4), None, batch_axis=0, **kw) as v:
            v.compute(lead)
            outs.append(v.read().array())
        kw = {"channel_axis": 0} if use_channel else {"sample_axis": 0}
        with ref.VizSession("lineplot", (4, 2), None, batch_axis=1, **kw) as v:
            v.compute(np.ascontiguousarray(lead.T))
            outs.append(v.read().array())
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])


def test_waterfall_port_matches_reference_ring(ref):
    """waterfall/module_tests.cc:186-217 (newest rows retained for arbitrary batch counts, height 5) and :262-333
    (2 * height + 2 batches twice: the cursor advances by batches % height)."""
    from oracle import port
    height, n = 5, 3
    p = port.Waterfall(n, height)
    next_value = 1.0
    sessions = {}
    for batches in (1, 5, 6, 10, 13, 3):
        x = (next_value + np.arange(batches * n, dtype=np.float32)).reshape(batches, n)
        next_value += batches * n
        # the reference module is created per input shape; the ring + cursor are carried by replaying into a fresh module
        # is not possible, so each batch count gets its own module fed the same history
        with ref.VizSession("waterfall", (batches, n), {"height": height}, sample_axis=1, batch_axis=0) as v:
            q = port.Waterfall(n, height)
            for _ in range(3):
                v.compute(x)
                q.compute(x)
                assert np.array_equal(v.read().array().reshape(height, n), q.ring) and v.write_index() == q.write_index
        p.compute(x)
    chrono = [p.ring[(p.write_index + r) % height] for r in range(height)]
    flat = np.concatenate(chrono)
    assert np.array_equal(flat, next_value - height * n + np.arange(height * n, dtype=np.float32))   # the newest 5 rows, in order
    x = (1.0 + np.arange(12 * 3, dtype=np.float32)).reshape(12, 3)
    with ref.VizSession("waterfall", (12, 3), {"height": 5}, sample_axis=1, batch_axis=0) as v:
        v.compute(x)
        assert v.write_index() == 2
        v.compute(x)
        assert v.write_index() == 4
