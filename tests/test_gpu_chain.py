"""GPU parity: fused spectral chain (b200_chain_exec through the host mirror) vs the reference CPU
spectrum_engine block run by the reference's own Flowgraph/scheduler (oracle/_ref)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from parity import assert_db_close, true_spectrum


def _window(n):
    from oracle import port
    return port.invert(port.window(n))          # the reference's taps, bit-exact (test_oracle), sign-flipped


def _run_chain(x, enable_scale, rmin=-120.0, rmax=0.0, fused=True):
    import cyberether_b200 as cb
    from cyberether_b200.blocks import SpectrumEngine
    block = SpectrumEngine(enableScale=enable_scale, rangeMin=rmin, rangeMax=rmax, fused=fused)
    inp = cb.Tensor.from_numpy(x, sampleAxis=x.ndim - 1, batchAxis=0 if x.ndim > 1 else None)
    assert block.create("spec", {"buffer": inp}) == cb.Result.SUCCESS, cb.last_error()
    for _ in range(2):
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
    out = block.output("buffer").numpy()
    block.destroy()
    return out


def _range_slope(rmin, rmax):
    return 2.0 / abs(rmax - rmin)   # max d(range)/d(dB): 0.5 * 4 * sech^2 <= 2, times 1/(max-min)


@pytest.mark.parametrize("rows", [1, 3, 64, 300])
def test_chain_4096_scale(ref, rows):
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(0, rows)
    want = ref.spectrum_engine(x, enable_scale=True)
    got = _run_chain(x, True)
    assert got.shape == want.shape and got.dtype == np.float32
    spec = true_spectrum(x, _window(4096))
    assert_db_close(got, want, spec, scale=_range_slope(-120.0, 0.0), floor=3e-7)


def test_chain_4096_db(ref):
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(1000, 128)
    want = ref.spectrum_engine(x, enable_scale=False)
    got = _run_chain(x, False)
    assert_db_close(got, want, true_spectrum(x, _window(4096)))


def test_chain_4096_unfused_modules_match_fused(ref):
    """The one-kernel-per-module wiring (reference's own module sequence on this provider) and the fused
    kernel agree with the reference to the same allowance."""
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(50, 32)
    want = ref.spectrum_engine(x, enable_scale=True)
    spec = true_spectrum(x, _window(4096))
    for fused in (False, True):
        got = _run_chain(x, True, fused=fused)
        assert_db_close(got, want, spec, scale=_range_slope(-120.0, 0.0), floor=3e-7)


def test_chain_sanity_golden():
    """BASELINE.md §2 golden: tone at bin 100, amplitude 0.5 -> peak bin 2148, -13.5583 dB, range 0.956732."""
    n = 4096
    x = (0.5 * np.exp(2j * np.pi * 100 * np.arange(n) / n)).astype(np.complex64)[None, :].repeat(4, 0)
    db = _run_chain(x, False)
    assert int(db[0].argmax()) == 2148
    assert abs(float(db[0].max()) - (-13.5583)) < 5e-4
    sc = _run_chain(x, True)
    assert abs(float(sc[0].max()) - 0.956732) < 5e-6


@pytest.mark.parametrize("n", [8, 64, 256, 1024, 2048, 8192, 16384, 32768, 65536])
def test_chain_other_sizes(ref, n):
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(7, 5, n=n)
    want = ref.spectrum_engine(x, enable_scale=True, range_min=-100.0, range_max=-10.0)
    got = _run_chain(x, True, -100.0, -10.0)
    assert_db_close(got, want, true_spectrum(x, _window(n)), scale=_range_slope(-100.0, -10.0), floor=3e-7)


@pytest.mark.parametrize("n", [16384, 65536])
def test_chain_tiled_two_pass_in_several_chunks_and_db_mode(ref, n, monkeypatch):
    """n = 16384 / 32768 / 65536: window multiply fused into the column pass, amplitude (/ range) into the row pass of the
    tiled two-pass plan (fft_tile.cuh). The chunk is forced down to 2 spectra so 5 spectra run as chunks of 2, 2, 1."""
    from cyberether_b200.synthetic import spectral_rows
    monkeypatch.setenv("B200_FFT_TWOPASS_CHUNK_MB", str(max(1, (2 * n * 8) >> 20)))
    x = spectral_rows(11, 5, n=n)
    spec = true_spectrum(x, _window(n))
    assert_db_close(_run_chain(x, False), ref.spectrum_engine(x, enable_scale=False), spec)
    want = ref.spectrum_engine(x, enable_scale=True, range_min=-90.0, range_max=-20.0)
    assert_db_close(_run_chain(x, True, -90.0, -20.0), want, spec, scale=_range_slope(-90.0, -20.0), floor=3e-7)
    zero = np.zeros((3, n), np.complex64)
    assert np.all(np.isneginf(_run_chain(zero, False)))
    assert ref.spectrum_engine(zero, enable_scale=True).equals(_run_chain(zero, True))


def test_chain_zero_input(ref):
    x = np.zeros((2, 4096), np.complex64)
    assert ref.spectrum_engine(x, enable_scale=True).equals(_run_chain(x, True))
    got = _run_chain(x, False)
    assert np.all(np.isneginf(got))
    want = ref.spectrum_engine(x, enable_scale=False)
    assert want.idx.size == want.size and np.all(np.isneginf(want.values))   # non-finite outputs are all stored


def test_chain_flat_range(ref):
    """min == max -> scale 0 -> constant 0.5 (src/domains/core/range/module_impl_native_cpu.cc:71-74)."""
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(3, 2)
    want = ref.spectrum_engine(x, enable_scale=True, range_min=-50.0, range_max=-50.0)
    got = _run_chain(x, True, -50.0, -50.0)
    assert want.equals(got) and np.all(got == 0.5)


def _chain_module(buffer, window, dtype=None, enable_scale=True, agc=False):
    import cyberether_b200 as cb
    ctx = cb.TestContext("spectral_chain")
    shape_rank = buffer.ndim - (1 if dtype and dtype.startswith("C") else 0)
    ctx.set_input("buffer", buffer, dtype=dtype, sampleAxis=shape_rank - 1, batchAxis=0 if shape_rank > 1 else None)
    ctx.set_input("window", window, sampleAxis=0)
    ctx.set_config(enableScale=enable_scale, rangeMin=-120.0, rangeMax=0.0, enableAgc=agc)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    return ctx.output("buffer")


@pytest.mark.parametrize("name,np_type,n,rows", [("CI8", np.int8, 4096, 300), ("CU8", np.uint8, 4096, 37),
                                                 ("CI16", np.int16, 4096, 300), ("CU16", np.uint16, 4096, 5),
                                                 ("CI32", np.int32, 4096, 9), ("CI8", np.int8, 1024, 40),
                                                 ("CI16", np.int16, 8192, 6)])
@pytest.mark.parametrize("enable_scale", [True, False])
def test_chain_integer_ingest_equals_cast_then_chain(ref, name, np_type, n, rows, enable_scale):
    """Fused complex-integer ingest (one kernel for n = 4096 / 8- and 16-bit samples, cast + chain otherwise):
    bit-identical to the provider's own cast module followed by the CF32 chain, and within the chain allowance of
    the reference's cast -> spectrum_engine flowgraph."""
    import cyberether_b200 as cb
    from oracle import port
    info = np.iinfo(np_type)
    rng = np.random.default_rng(n + rows)
    # a few tones + noise, quantised to the integer range (an SDR capture)
    t = np.arange(n)
    sig = sum(a * np.exp(2j * np.pi * f * t / n) for a, f in [(0.5, 100.25), (0.05, 1500.5), (0.002, 3000.0)])
    sig = sig[None, :] * np.exp(2j * np.pi * rng.random((rows, 1))) + 0.01 * (rng.standard_normal((rows, n)) +
                                                                              1j * rng.standard_normal((rows, n)))
    half = (float(info.max) - float(info.min) + 1) / 2
    mid = 0.0 if info.min < 0 else half
    x = np.stack([sig.real, sig.imag], axis=-1) * half * 0.9 + mid
    x = np.clip(np.rint(x), info.min, info.max).astype(np_type)
    w = _window(n)
    got = _chain_module(x, w, dtype=name, enable_scale=enable_scale)
    xf = port.cast(x, complex_pairs=True)                    # bit-exact restatement of the reference cast (test_oracle)
    two_step = _chain_module(xf, w, enable_scale=enable_scale)
    assert got.shape == (rows, n) and got.dtype == np.float32
    assert np.array_equal(got, two_step)
    with ref.Session() as s:
        s.add_source("src", x, sample_axis=1, batch_axis=0, dtype=name)
        s.add_block("c", "cast", {"outputType": "CF32"}, {"buffer": "src.signal"})
        s.add_block("se", "spectrum_engine", {"enableScale": enable_scale, "rangeMin": -120.0, "rangeMax": 0.0},
                    {"buffer": "c.buffer"})
        s.compute()
        s.compute()
        want = s.output("se", "buffer")
    spec = true_spectrum(xf, w)
    if enable_scale:
        assert_db_close(got, want, spec, scale=_range_slope(-120.0, 0.0), floor=3e-7)
    else:
        assert_db_close(got, want, spec)


@pytest.mark.parametrize("enable_scale", [True, False])
@pytest.mark.parametrize("fused", [True, False])
@pytest.mark.parametrize("n,level", [(4096, 0.03), (4096, 30.0), (4096, 1e-4), (1024, 0.03)])
def test_spectrum_engine_with_agc(ref, enable_scale, fused, n, level):
    """enableAgc: an `agc` module (one RMS tile per spectrum) between fft and amplitude (block_impl.cc:186-200).
    4096-point spectra run it inside the fused kernel (row power by Parseval), other lengths and fused=False module by
    module. Levels: gain inside its clamp range, clamped at minGain (loud) and at maxGain (quiet)."""
    import cyberether_b200 as cb
    from cyberether_b200.blocks import SpectrumEngine
    from cyberether_b200.synthetic import spectral_rows
    x = spectral_rows(7, 48, n=n) * np.float32(level)
    block = SpectrumEngine(enableAgc=True, enableScale=enable_scale, fused=fused)
    inp = cb.Tensor.from_numpy(x, sampleAxis=1, batchAxis=0)
    assert block.create("spec", {"buffer": inp}) == cb.Result.SUCCESS, cb.last_error()
    for _ in range(2):
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
    got = block.output("buffer").numpy()
    assert ("spectral_chain" in block.modules) == (fused and n == 4096)
    assert ("agc" in block.modules) != ("spectral_chain" in block.modules)
    block.destroy()
    want = ref.run_block("spectrum_engine", {"buffer": x}, {"enableAgc": True, "enableScale": enable_scale,
                                                           "rangeMin": -120.0, "rangeMax": 0.0}, "buffer")
    # the gain is common to a row: the allowance is computed on the spectrum the amplitude stage sees (g X)
    w = _window(n)
    spec = true_spectrum(x, w)
    mean_power = (np.abs(spec) ** 2).mean(axis=1, keepdims=True)
    gain = np.clip(1.0 / np.sqrt(mean_power + 1e-12), 0.01, 100.0)
    if enable_scale:
        assert_db_close(got, want, spec * gain, scale=_range_slope(-120.0, 0.0), floor=3e-7)
    else:
        assert_db_close(got, want, spec * gain)


@pytest.mark.parametrize("name,np_type", [("CI8", np.int8), ("CU16", np.uint16)])
def test_chain_integer_ingest_with_agc(name, np_type):
    """Integer ingest and the AGC stage in the same kernel: bit-identical to cast -> CF32 chain with AGC."""
    from oracle import port
    info = np.iinfo(np_type)
    x = np.random.default_rng(11).integers(info.min // 4, info.max // 4, size=(33, 4096, 2), dtype=np_type)
    w = _window(4096)
    got = _chain_module(x, w, dtype=name, agc=True)
    two_step = _chain_module(port.cast(x, complex_pairs=True), w, agc=True)
    assert np.array_equal(got, two_step)
    assert not np.array_equal(got, _chain_module(x, w, dtype=name, agc=False))


def test_chain_full_size_rows_are_independent(ref):
    """BASELINE configs[1] at full size (65536 x 4096, 2 GiB in / 1 GiB out) through the C ABI: rows of the big launch
    (221 rows per persistent CTA, TMA ring wrapped ~74 times) are bit-identical to the same rows processed in a 64-row
    launch, and 1024 rows spread over the whole batch (every 64th) are checked against the REFERENCE itself (the round-1
    version compared 8 rows with the reference)."""
    import ctypes
    import torch
    import cyberether_b200 as cb
    from cyberether_b200 import _native
    from cyberether_b200.jetstream import Context
    from cyberether_b200.synthetic import spectral_rows
    lib = _native.load()
    dev = torch.device("cuda:0")
    ctx = Context.get(dev)
    rows, n = 65536, 4096
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234)
    x = torch.view_as_complex(torch.randn(rows, n, 2, device=dev, generator=gen) * 0.01)
    picks = [0, 1, 147, 295, 296, 591, 592, 32767, 32768, 65534, 65535] + [int(v) for v in
             np.random.default_rng(5).integers(0, rows, 53)]
    small_in = torch.from_numpy(spectral_rows(0, 64)).to(dev)
    x[torch.tensor(picks[:8], device=dev)] = small_in[:8]              # a few rows the reference has seen
    win = torch.from_numpy(_window(n)).to(dev)
    coeff = cb.amplitude_scaling_coeff(n)
    sc, off = cb.range_coefficients(-120.0, 0.0)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    plan = ctypes.c_void_p()
    _native.check(lib.b200_chain_plan_create(ctx.handle, n, rows, win.data_ptr(), ctypes.byref(plan)))
    big = torch.empty(rows, n, dtype=torch.float32, device=dev)
    _native.check(lib.b200_chain_exec(plan, x.data_ptr(), big.data_ptr(), rows, coeff, 1, sc, off, stream))
    sub_in = x[torch.tensor(picks, device=dev)].contiguous()
    sub = torch.empty(len(picks), n, dtype=torch.float32, device=dev)
    _native.check(lib.b200_chain_exec(plan, sub_in.data_ptr(), sub.data_ptr(), len(picks), coeff, 1, sc, off, stream))
    torch.cuda.synchronize()
    _native.check(lib.b200_chain_plan_destroy(plan))
    assert torch.equal(big[torch.tensor(picks, device=dev)], sub)
    assert bool(torch.isfinite(big).all()) and float(big.min()) >= 0.0 and float(big.max()) <= 1.0
    want = ref.spectrum_engine(spectral_rows(0, 8), enable_scale=True)
    spec = true_spectrum(spectral_rows(0, 8), _window(n))
    assert_db_close(sub[:8].cpu().numpy(), want, spec, scale=_range_slope(-120.0, 0.0), floor=3e-7)
    # 1024 rows of the big launch against the reference CPU block (Gaussian rows: every bin is a "strong" bin)
    stride_rows = torch.arange(0, rows, 64, device=dev)
    x_host = x[stride_rows].cpu().numpy()
    want_many = ref.spectrum_engine(x_host, enable_scale=True)
    from parity import assert_strong_bins
    spec_many = true_spectrum(x_host, _window(n))
    got_many = big[stride_rows].cpu().numpy()
    assert_db_close(got_many, want_many, spec_many, scale=_range_slope(-120.0, 0.0), floor=3e-7)
    assert_strong_bins(got_many, want_many, spec_many, slope=_range_slope(-120.0, 0.0), label="full-size rows")
    # every element of the 1024 rows: against the numpy restatement of the reference chain (another FP32 FFT)
    from oracle import port
    whole = port.spectrum_engine(x_host, enable_scale=True)
    assert_db_close(got_many, whole, spec_many, scale=_range_slope(-120.0, 0.0), floor=3e-7)
    assert_strong_bins(got_many, whole, spec_many, slope=_range_slope(-120.0, 0.0), label="full-size rows vs port")
