"""GPU parity of the standalone modules (one C-ABI call each, through the host mirror's TestContext) against
the reference CPU modules (oracle/_ref), plus the reference's own known-answer cases restated
(src/domains/**/module_tests.cc, SURVEY.md §4)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(module_type, inputs, config=None, out="signal", axes=None):
    import cyberether_b200 as cb
    ctx = cb.TestContext(module_type)
    for name, arr in inputs.items():
        ax = (axes or {}).get(name)
        if ax is None:
            ax = dict(sampleAxis=arr.ndim - 1, batchAxis=0 if arr.ndim > 1 else None)
        ctx.set_input(name, arr, **ax)
    ctx.set_config(**(config or {}))
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    return ctx.output(out)


@pytest.mark.parametrize("n", [1, 2, 7, 8, 1000, 1024, 4096, 65536])
def test_window_matches_reference(ref, n):
    got = _run("window", {}, {"size": n}, out="window")
    want = ref.window(n)
    assert got.dtype == np.complex64 and got.shape == want.shape == (n,)
    # F64 cos on the device vs glibc: identical after rounding to F32 except for rare double-rounding ties.
    g, w = want.take(got), want.values
    ulp = np.spacing(np.abs(w.real).astype(np.float32)).max()
    assert np.abs(g.real - w.real).max() <= ulp
    assert np.all(got.imag == 0)
    assert float((g.real != w.real).mean()) < 1e-3


def test_window_formula_known_answer():
    """src/domains/dsp/window/module_tests.cc:45 — taps match the Blackman formula within 1e-5."""
    n = 64
    got = _run("window", {}, {"size": n}, out="window")
    i = np.arange(n)
    want = 0.42 - 0.5 * np.cos(2 * np.pi * i / (n - 1)) + 0.08 * np.cos(4 * np.pi * i / (n - 1))
    assert np.abs(got.real - want).max() < 1e-5


@pytest.mark.parametrize("shape,axis", [((4096,), 0), ((8, 64), 1), ((5, 7), 1), ((3, 4, 6), 2)])
def test_invert_bit_exact(ref, shape, axis):
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32(shape, 11)
    got = _run("invert", {"signal": x})
    want = ref.run_block("invert", {"signal": x}, None, "signal")
    if shape[axis] % 2 == 0:
        assert want.equals(got)                   # sign flips are exact
        from oracle import port                   # the whole output: the restatement pinned to the reference
        assert np.array_equal(got, port.invert(x, axis))
    else:
        assert np.abs(want.diff(got)).max() <= 2 * np.spacing(np.float32(want.absmax()))


@pytest.mark.parametrize("sa,sb", [((64, 4096), (1, 4096)), ((64, 4096), (64, 4096)), ((4, 3, 8), (3, 1)),
                                   ((16,), (16,)), ((2, 5), (5,)), ((6, 1, 4), (1, 7, 1))])
def test_multiply_cf32_bit_exact(ref, sa, sb):
    from cyberether_b200.synthetic import gaussian_cf32
    a, b = gaussian_cf32(sa, 1), gaussian_cf32(sb, 2)
    # only the sample axis is declared (right-aligned roles must agree, src/memory/axis.cc:332-359)
    axes = {"a": dict(sampleAxis=len(sa) - 1), "b": dict(sampleAxis=len(sb) - 1)}
    got = _run("multiply", {"a": a, "b": b}, out="product", axes=axes)
    want = ref.run_block("multiply", {"a": a, "b": b}, None, "product",
                         axes={"a": (len(sa) - 1, -1, -1), "b": (len(sb) - 1, -1, -1)})
    assert got.shape == want.shape
    assert want.equals(got)
    from oracle import port                       # the whole output: the restatement pinned to the reference
    assert np.array_equal(got, port.multiply(a, b))


def test_multiply_conflicting_axes_rejected_like_reference(ref):
    """Batch roles that right-align to different output axes are an ERROR in the reference
    ("Signal roles map to conflicting output axes"); the mirror rejects the same graph."""
    import cyberether_b200 as cb
    from cyberether_b200.synthetic import gaussian_cf32
    a, b = gaussian_cf32((4, 3, 8), 1), gaussian_cf32((3, 1), 2)
    with pytest.raises(ref.RefError):
        ref.run_block("multiply", {"a": a, "b": b}, None, "product", axes={"a": (2, 0, -1), "b": (1, 0, -1)})
    ctx = cb.TestContext("multiply")
    ctx.set_input("a", a, sampleAxis=2, batchAxis=0)
    ctx.set_input("b", b, sampleAxis=1, batchAxis=0)
    assert ctx.run() == cb.Result.ERROR
    assert "conflicting output axes" in cb.last_error()


def test_multiply_f32_bit_exact(ref):
    rng = np.random.default_rng(3)
    a = rng.standard_normal((128, 512)).astype(np.float32)
    b = rng.standard_normal((512,)).astype(np.float32)
    from oracle import port
    got = _run("multiply", {"a": a, "b": b}, out="product")
    assert ref.multiply(a, b).equals(got) and np.array_equal(got, port.multiply(a, b))


@pytest.mark.parametrize("n", [2, 4, 8, 16, 32, 64, 128, 256, 512, 1024, 2048, 4096, 8192, 16384])
@pytest.mark.parametrize("forward", [True, False])
def test_fft_c2c_matches_reference(ref, n, forward):
    """North-star tolerance for the spectrum: max|a-b| <= 1e-5 * max|b| per transform (we assert 2e-6)."""
    from cyberether_b200.synthetic import gaussian_cf32
    rows = 7 if n <= 4096 else 3
    x = gaussian_cf32((rows, n), 100 + n)
    got = _run("fft", {"signal": x}, {"forward": forward})
    want = ref.fft(x, forward=forward)
    rel = np.abs(want.diff(got)) / want.row_absmax_at()
    assert rel.max() <= 2e-6, rel.max()
    exact = np.fft.fft(x.astype(np.complex128), axis=-1) if forward else np.fft.ifft(x.astype(np.complex128), axis=-1) * n
    ours = np.abs(want.diff(got) - (want.take(exact) - want.values)).max() / np.abs(exact).max()
    theirs = np.abs(want.values - want.take(exact)).max() / np.abs(exact).max()
    assert ours <= 3 * theirs + 1e-7, (ours, theirs)    # no less accurate than pocketfft


def test_fft_4096_large_batch_roundtrip():
    """Size-independent property at scale: ifft(fft(x)) == N x (reference fft/module_tests.cc:136-143)."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((2048, 4096), 5)
    y = _run("fft", {"signal": x}, {"forward": True})
    z = _run("fft", {"signal": y}, {"forward": False})
    assert np.abs(z / 4096 - x).max() <= 1e-5 * np.abs(x).max()


def test_fft_known_answers():
    """fft/module_tests.cc: DC -> spike at bin 0 (1e-3), single tone -> spike at its bin."""
    n = 64
    got = _run("fft", {"signal": np.ones(n, np.complex64)}, {"forward": True})
    assert abs(got[0].real - n) < 1e-3 and np.abs(got[1:]).max() < 1e-3
    n = 1024
    x = np.exp(2j * np.pi * 5 * np.arange(n) / n).astype(np.complex64)
    got = _run("fft", {"signal": x}, {"forward": True})
    assert abs(abs(got[5]) - 1024.0) < 1e-2 and int(np.abs(got).argmax()) == 5


def test_amplitude_cf32_bit_exact(ref):
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((32, 4096), 9, scale=30.0)
    x[0, :8] = 0
    x[1, :4] = [1e-30, 1e30, 1 + 0j, 2 + 0j]
    got = _run("amplitude", {"signal": x})
    want = ref.amplitude(x)
    assert want.equals(got)                       # same operation order, no FMA: bit-identical
    from oracle import port
    assert np.array_equal(got, port.amplitude(x, 4096))
    assert np.all(np.isneginf(got[0, :8]))


def test_amplitude_f32_bit_exact(ref):
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((16, 1000)) * 10).astype(np.float32)
    x[0, 0] = 0.0
    from oracle import port
    got = _run("amplitude", {"signal": x})
    assert ref.amplitude(x).equals(got) and np.array_equal(got, port.amplitude(x, 1000))


@pytest.mark.parametrize("lo,hi", [(-1.0, 1.0), (-120.0, 0.0), (0.0, -120.0), (5.0, 5.0)])
def test_range_matches_reference(ref, lo, hi):
    rng = np.random.default_rng(5)
    x = (rng.standard_normal((64, 1024)) * max(1.0, abs(hi - lo))).astype(np.float32)
    x[0, :3] = [-np.inf, np.inf, 0.0]
    got = _run("range", {"signal": x}, {"min": lo, "max": hi})
    want = ref.range_(x, lo, hi)
    # CUDA tanhf vs glibc tanhf: <= 2 ulp of tanh -> <= 1.2e-7 absolute on [0, 1] (reference test: 1e-6).
    assert np.abs(want.diff(got)).max() <= 2.5e-7
    assert np.array_equal(got.reshape(-1)[want.idx[:2]], want.values[:2]) and want.idx[1] == 1     # -inf and inf


def test_cast_bypass_and_f32():
    import cyberether_b200 as cb
    x = np.arange(8, dtype=np.float32)
    got = _run("cast", {"buffer": x}, {"outputType": "CF32"}, out="buffer")
    assert np.array_equal(got, x.astype(np.complex64))


# ---- DISCONTIGUOUS layouts (reference: "Trailing Batch Strided", "Rank 3 Batched Heads", "Rank 4 Non-Contiguous") ----

def _run_view(module_type, base, view_fn, axes, config=None, out="signal"):
    """Feeds a strided/permuted torch VIEW of `base` (so the module really sees a non-contiguous tensor)."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.jetstream import TensorLink, NativeCudaRuntime
    dev = torch.from_numpy(base).cuda()
    tensor = cb.Tensor(view_fn(dev), dict(axes))
    module = cb.build_module(module_type)
    assert module.create("dut", config, {"signal": TensorLink(tensor=tensor)}) == cb.Result.SUCCESS, cb.last_error()
    rt = NativeCudaRuntime("t")
    assert rt.create([module]) == cb.Result.SUCCESS
    assert rt.compute([], set(), set()) == cb.Result.SUCCESS, cb.last_error()
    result = module.outputs[out].tensor.numpy()
    rt.destroy()
    module.destroy()
    return result


def test_fft_trailing_batch_axis(ref):
    """Sample axis 0, batch axis 1 ("FFT - Trailing Batch Roundtrip CF32", fft/module_tests.cc:802-852)."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((256, 6), 21)
    want = ref.run_block("fft", {"signal": x}, {"forward": True}, "signal", axes={"signal": (0, 1, -1)})
    got = _run_view("fft", x, lambda t: t, {"sampleAxis": 0, "batchAxis": 1}, {"forward": True})
    assert got.shape == want.shape
    assert np.abs(want.diff(got)).max() <= 2e-6 * want.absmax()


def test_fft_rank3_heads_middle_sample_axis(ref):
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((3, 128, 5), 22)
    want = ref.run_block("fft", {"signal": x}, {"forward": False}, "signal", axes={"signal": (1, 0, 2)})
    got = _run_view("fft", x, lambda t: t, {"sampleAxis": 1, "batchAxis": 0, "channelAxis": 2}, {"forward": False})
    assert np.abs(want.diff(got)).max() <= 2e-6 * want.absmax()


def test_fft_strided_slice_view():
    """A strided view (every other row of a larger buffer, offset start) transforms like its dense copy."""
    from cyberether_b200.synthetic import gaussian_cf32
    base = gaussian_cf32((10, 512), 23)
    got = _run_view("fft", base, lambda t: t[1::2, :], {"sampleAxis": 1, "batchAxis": 0}, {"forward": True})
    want = np.fft.fft(base[1::2, :].astype(np.complex128), axis=1)
    assert got.shape == (5, 512)
    assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max()


def test_amplitude_and_range_non_contiguous_bit_exact(ref):
    from cyberether_b200.synthetic import gaussian_cf32
    base = gaussian_cf32((4, 6, 64), 24, 5.0)
    view = np.ascontiguousarray(base.transpose(1, 0, 2)[:, ::2, :])          # dense copy of what the view holds
    got = _run_view("amplitude", base, lambda t: t.permute(1, 0, 2)[:, ::2, :], {"sampleAxis": 2})
    want = ref.run_block("amplitude", {"signal": view}, None, "signal", axes={"signal": (2, -1, -1)})
    assert want.equals(got)
    fbase = np.random.default_rng(1).standard_normal((6, 40)).astype(np.float32)
    got = _run_view("range", fbase, lambda t: t[:, ::4], {}, {"min": -2.0, "max": 2.0})
    want = ref.range_(np.ascontiguousarray(fbase[:, ::4]), -2.0, 2.0)
    assert np.abs(want.diff(got)).max() <= 2.5e-7


# ---- real-input transforms ("FFT - Complex Real Signal F32", "FFT - FFTPACK Real ...", fft/module_tests.cc:149-440) ----

@pytest.mark.parametrize("shape,axes", [((256,), (0, -1, -1)), ((6, 1024), (1, 0, -1)), ((64, 5), (0, 1, -1))])
def test_fft_r2c_complex_output(ref, shape, axes):
    rng = np.random.default_rng(31)
    x = rng.standard_normal(shape).astype(np.float32)
    want = ref.run_block("fft", {"signal": x}, {"forward": True, "complexOutput": True}, "signal", axes={"signal": axes})
    names = dict(zip(("sampleAxis", "batchAxis", "channelAxis"), [a if a >= 0 else None for a in axes]))
    got = _run_view("fft", x, lambda t: t, {k: v for k, v in names.items() if v is not None},
                    {"forward": True, "complexOutput": True})
    assert got.shape == want.shape and got.dtype == np.complex64
    assert np.abs(want.diff(got)).max() <= 2e-6 * want.absmax()


@pytest.mark.parametrize("n", [8, 64, 2048])
def test_fft_fftpack_real_forward_inverse(ref, n):
    rng = np.random.default_rng(32)
    x = rng.standard_normal((4, n)).astype(np.float32)
    half_complex = rng.standard_normal((4, n)).astype(np.float32)        # any real row is an FFTPACK spectrum
    fwd_want = ref.run_block("fft", {"signal": x}, {"forward": True}, "signal")
    inv_want = ref.run_block("fft", {"signal": half_complex}, {"forward": False}, "signal")
    fwd = _run("fft", {"signal": x}, {"forward": True})
    assert fwd.dtype == np.float32 and fwd.shape == (4, n)
    assert np.abs(fwd_want.diff(fwd)).max() <= 2e-6 * fwd_want.absmax()
    inv = _run("fft", {"signal": half_complex}, {"forward": False})
    assert np.abs(inv_want.diff(inv)).max() <= 2e-6 * inv_want.absmax()
    inv = _run("fft", {"signal": fwd}, {"forward": False})
    assert np.abs(inv / n - x).max() <= 1e-5          # unnormalised round trip (reference tolerance 1e-2)


@pytest.mark.parametrize("n", [16384, 32768, 65536])
def test_fft_large_power_of_two_four_step(ref, n):
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((3, n), n)
    for forward in (True, False):
        got = _run("fft", {"signal": x}, {"forward": forward})
        want = ref.fft(x, forward=forward)
        assert np.abs(want.diff(got)).max() <= 3e-6 * want.absmax()


@pytest.mark.parametrize("n", [3, 5, 7, 12, 100, 1000, 4095, 4099, 8320])
def test_fft_arbitrary_length_bluestein(ref, n):
    """Non-power-of-two lengths (8320 = 8192 + 128 is what the reference's filter block feeds its fft)."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((4, n), 7 * n)
    for forward in (True, False):
        got = _run("fft", {"signal": x}, {"forward": forward})
        want = ref.fft(x, forward=forward)
        assert np.abs(want.diff(got)).max() <= 1e-5 * want.absmax()     # north-star tolerance


def test_chain_non_power_of_two_length(ref):
    import sys, os
    sys.path.insert(0, os.path.dirname(__file__))
    from parity import assert_db_close, true_spectrum
    import cyberether_b200 as cb
    from cyberether_b200.blocks import SpectrumEngine
    from cyberether_b200.synthetic import spectral_rows
    n = 1000
    x = spectral_rows(3, 6, n=n)
    want = ref.spectrum_engine(x, enable_scale=True)
    block = SpectrumEngine(enableScale=True)
    assert block.create("s", {"buffer": cb.Tensor.from_numpy(x, sampleAxis=1, batchAxis=0)}) == cb.Result.SUCCESS
    assert block.compute() == cb.Result.SUCCESS, cb.last_error()
    got = block.output("buffer").numpy()
    block.destroy()
    from oracle import port
    w = port.invert(port.window(n))
    assert_db_close(got, want, true_spectrum(x, w), scale=2.0 / 120.0, floor=3e-7)


CAST_CASES = [("I8", np.int8, False), ("U8", np.uint8, False), ("I16", np.int16, False), ("U16", np.uint16, False),
              ("I32", np.int32, False), ("U32", np.uint32, False), ("CI8", np.int8, True), ("CU8", np.uint8, True),
              ("CI16", np.int16, True), ("CU16", np.uint16, True), ("CI32", np.int32, True), ("CU32", np.uint32, True)]


@pytest.mark.parametrize("name,np_type,is_complex", CAST_CASES)
@pytest.mark.parametrize("shape", [(1,), (5, 37), (3, 4096)])
def test_cast_integer_bit_exact(ref, name, np_type, is_complex, shape):
    """cast: every integer / complex-integer conversion of the reference's native module, bit-exact, including the
    extreme values and sizes that exercise the vector body and the scalar tail."""
    import zlib
    import cyberether_b200 as cb
    info = np.iinfo(np_type)
    rng = np.random.default_rng(zlib.crc32(name.encode()) % 1000)       # the same input in every process
    full = shape + (2,) if is_complex else shape
    x = rng.integers(info.min, info.max, size=full, endpoint=True, dtype=np_type)
    x.flat[0] = info.min
    x.flat[-1] = info.max
    out_type = "CF32" if is_complex else "F32"
    want = ref.run_block("cast", {"buffer": x}, {"outputType": out_type}, "buffer", dtypes={"buffer": name})
    ctx = cb.TestContext("cast")
    ctx.set_input("buffer", x, dtype=name, sampleAxis=len(shape) - 1)
    ctx.set_config(outputType=out_type)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    got = ctx.output("buffer")
    assert got.dtype == want.dtype and got.shape == want.shape == shape
    assert want.equals(got)
    from oracle import port                       # the whole output: the restatement pinned to the reference
    assert np.array_equal(got, port.cast(x, complex_pairs=is_complex))


def test_cast_unsupported_pair_is_an_error():
    import cyberether_b200 as cb
    ctx = cb.TestContext("cast")
    ctx.set_input("buffer", np.zeros((4, 2), np.int8), dtype="CI8", sampleAxis=0)
    ctx.set_config(outputType="F32")                       # complex integer -> real float is not a reference pair
    assert ctx.run() == cb.Result.ERROR
    assert "Unsupported conversion" in cb.last_error()


def _assert_agc_equal(got, want):
    """Gains are F64 on both sides and differ only by the order of the F64 power sum (a few F64 ulp), so the F32
    outputs are identical except for rare last-bit rounding flips."""
    assert got.shape == want.shape and got.dtype == want.dtype
    if hasattr(want, "row_absmax"):                 # a stored sample of the reference output
        got, want = want.take(got), want.values
    g = got.view(np.float32) if np.iscomplexobj(got) else got
    w = want.view(np.float32) if np.iscomplexobj(want) else want
    both_nan = np.isnan(g) & np.isnan(w)
    diff = (g != w) & ~both_nan
    assert float(diff.mean()) <= 1e-4, f"{int(diff.sum())} of {diff.size} values differ"
    if diff.any():
        assert np.all(np.abs(g[diff] - w[diff]) <= np.spacing(np.abs(w[diff])))


@pytest.mark.parametrize("complex_input", [True, False])
@pytest.mark.parametrize("shape,tile,axis", [((3, 1000), 256, 1), ((64, 4096), 4096, 1), ((1, 77), 1024, 1),
                                             ((4, 5000), 64, 1), ((300, 6), 4, 0), ((2, 3, 520), 128, 2)])
def test_agc_matches_reference(ref, complex_input, shape, tile, axis):
    """agc module vs the reference's agc block (parameters chosen exactly representable in F32, because the
    reference BLOCK stores them as F32) and vs the pinned numpy restatement with the module's F64 defaults."""
    import cyberether_b200 as cb
    from oracle import port
    rng = np.random.default_rng(sum(shape) + tile)
    n = shape[axis]
    env_shape = [1] * len(shape)
    env_shape[axis] = n
    step = (1 + 7 * (np.arange(n) > n // 2)).reshape(env_shape)             # a level jump the rate limit must follow
    lane_shape = [s if d != axis else 1 for d, s in enumerate(shape)]
    env = np.exp(rng.uniform(-6, 6, size=lane_shape)) * step
    x = rng.standard_normal(shape) * env
    x = (x + 1j * rng.standard_normal(shape) * env).astype(np.complex64) if complex_input else x.astype(np.float32)
    axes = dict(sampleAxis=axis, batchAxis=None)
    exact = dict(tileSize=tile, reference=0.5, epsilon=2.0 ** -40, minGain=0.0625, maxGain=64.0, maxGainChange=2.0)
    ctx = cb.TestContext("agc")
    ctx.set_input("signal", x, **axes)
    ctx.set_config(**exact)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    want = ref.run_block("agc", {"signal": x}, exact, "signal", axes={"signal": (axis, -1, -1)})
    _assert_agc_equal(ctx.output("signal"), want)
    ctx = cb.TestContext("agc")
    ctx.set_input("signal", x, **axes)
    ctx.set_config(tileSize=tile)                                             # module defaults (F64 0.01, 1e-12, ...)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    _assert_agc_equal(ctx.output("signal"), port.agc(x, tile_size=tile, axis=axis))


def test_agc_keeps_huge_inputs_finite_like_reference(ref):
    """ApplyGain limits every product to the finite F32 range (module_impl_native_cpu.cc:36-60)."""
    import cyberether_b200 as cb
    big = np.float32(3.0e38)
    x = np.zeros((2, 512), np.complex64)
    x[0, :] = 1e-3
    x[0, 100] = big + 1j * big            # |z| beyond FLT_MAX
    x[1, :] = (np.arange(512) % 7) * 1e-3
    x[1, 5] = -big
    cfg = dict(tileSize=128, reference=1.0, epsilon=2.0 ** -40, minGain=0.5, maxGain=64.0, maxGainChange=4.0)
    ctx = cb.TestContext("agc")
    ctx.set_input("signal", x, sampleAxis=1, batchAxis=0)
    ctx.set_config(**cfg)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    got = ctx.output("signal")
    want = ref.run_block("agc", {"signal": x}, cfg, "signal")
    assert np.all(np.isfinite(got.view(np.float32)))
    _assert_agc_equal(got, want)


def test_agc_rejects_bad_config_like_reference():
    import cyberether_b200 as cb
    for bad, text in ((dict(tileSize=0), "Tile size"), (dict(reference=0.0), "Reference"),
                      (dict(minGain=2.0, maxGain=1.0), "Maximum gain"), (dict(maxGainChange=0.5), "gain change")):
        ctx = cb.TestContext("agc")
        ctx.set_input("signal", np.ones((2, 8), np.float32), sampleAxis=1, batchAxis=0)
        ctx.set_config(**bad)
        assert ctx.run() == cb.Result.ERROR
        assert text in cb.last_error()


def test_cast_non_contiguous_view_like_reference_test():
    """core/cast/module_tests.cc:628-668 — a sliced + permuted I8 view (non-zero offset, not contiguous) -> F32."""
    import torch
    import cyberether_b200 as cb
    storage = (np.arange(24, dtype=np.int64) - 12).astype(np.int8).reshape(2, 3, 4)
    dev = torch.from_numpy(storage).cuda()
    view = dev[1].permute(1, 0)                       # shape (4, 3), offset 12, strides (1, 4)
    assert not view.is_contiguous() and view.storage_offset() != 0
    t = cb.Tensor(view)
    t.set_attribute("sampleAxis", 1)
    link = cb.TensorLink()
    link.produced("test", "buffer", t)
    module = cb.build_module("cast", "cuda", "native", "b200")
    assert module.create("cast", {"outputType": "F32"}, {"buffer": link}) == cb.Result.SUCCESS, cb.last_error()
    runtime = cb.NativeCudaRuntime("test", "cuda")
    assert runtime.create([module]) == cb.Result.SUCCESS
    assert runtime.compute([], set(), set()) == cb.Result.SUCCESS, cb.last_error()
    out = module.outputs["buffer"].tensor.numpy()
    want = storage[1].T.astype(np.float32) / np.float32(128.0)
    assert out.shape == (4, 3) and np.array_equal(out, want)
    runtime.destroy()
    module.destroy()


@pytest.mark.parametrize("name,np_type,is_complex", CAST_CASES + [("F32", np.float32, False)])
def test_cast_matching_dtype_is_a_bypass(name, np_type, is_complex):
    """core/cast/module_tests.cc "preserves every matching dtype bypass": the output aliases the input."""
    import cyberether_b200 as cb
    x = np.ones((3, 2) if is_complex else (3,), np_type)
    ctx = cb.TestContext("cast")
    ctx.set_input("buffer", x, dtype=name if name != "F32" else None, sampleAxis=0)
    ctx.set_config(outputType=name)
    assert ctx.start() == cb.Result.SUCCESS, cb.last_error()
    assert ctx.module.bypass
    assert ctx.module.outputs["buffer"].tensor.data.data_ptr() == ctx.inputs["buffer"].data.data_ptr()
    assert ctx.compute() == cb.Result.SUCCESS
    ctx.stop()


@pytest.mark.parametrize("spelling", ["", "cf32", "CF32 ", "NONE", "NOPE"])
def test_cast_rejects_invalid_output_spelling(spelling):
    """core/cast/module_tests.cc:670-686."""
    import cyberether_b200 as cb
    ctx = cb.TestContext("cast")
    ctx.set_input("buffer", np.zeros((2, 2), np.int8), dtype="CI8", sampleAxis=0)
    ctx.set_config(outputType=spelling)
    assert ctx.run() == cb.Result.ERROR
    assert "Invalid output type" in cb.last_error()


@pytest.mark.parametrize("complex_input", [True, False])
@pytest.mark.parametrize("lanes,samples,tile", [(600, 3000, 1024), (400, 4096, 4096), (320, 777, 256), (512, 2048, 2048)])
def test_agc_fused_one_cta_per_lane_form(ref, complex_input, lanes, samples, tile):
    """agc_fused_kernel (enough lanes to fill the GPU, tiles that fit one CTA's registers): every sample read once, the
    tile kept in registers between its power sum and its apply. Against the numpy restatement of the reference and the
    three-kernel form; a level jump per lane exercises the rate limit, the last tile is ragged."""
    import cyberether_b200 as cb
    from oracle import port
    rng = np.random.default_rng(lanes + samples + tile)
    step = 1 + 7 * (np.arange(samples) > samples // 2)[None, :]
    env = np.exp(rng.uniform(-6, 6, size=(lanes, 1))) * step
    x = rng.standard_normal((lanes, samples)) * env
    x = (x + 1j * rng.standard_normal((lanes, samples)) * env).astype(np.complex64) if complex_input else x.astype(np.float32)

    def run():
        ctx = cb.TestContext("agc")
        ctx.set_input("signal", x, sampleAxis=1, batchAxis=0)
        ctx.set_config(tileSize=tile)
        assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
        return ctx.output("signal")
    results = {}
    for mode in ("1", "0"):              # 1: fused form up to 16 samples per thread, 0: three kernels
        os.environ["B200_AGC_FUSED"] = mode
        try:
            results[mode] = run()
        finally:
            del os.environ["B200_AGC_FUSED"]
    fused, three = results["1"], results["0"]
    want = port.agc(x, tile_size=tile, axis=1)
    _assert_agc_equal(fused, want)
    _assert_agc_equal(three, want)
    _assert_agc_equal(fused, three)
