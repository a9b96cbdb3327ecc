"""GPU parity for the `filter` block (fused streaming FIR) and the `fm` module against the reference CPU
blocks run by the reference's own Flowgraph (oracle/_ref), including state carried across compute cycles."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _ref_filter(ref, cycles, config):
    outs = []
    with ref.Session() as s:
        s.add_source("src", cycles[0], sample_axis=cycles[0].ndim - 1, batch_axis=0 if cycles[0].ndim > 1 else -1)
        s.add_block("flt", "filter", config, {"signal": "src.signal"})
        for x in cycles:
            s.write_source("src", x)
            s.compute()
            outs.append(s.output("flt", "buffer"))
        info = s.output_info("flt", "buffer")
    return outs, info


def _our_filter(cycles, config):
    import cyberether_b200 as cb
    from cyberether_b200.blocks import Filter
    x0 = cycles[0]
    inp = cb.Tensor.from_numpy(x0, sampleAxis=x0.ndim - 1, batchAxis=0 if x0.ndim > 1 else None)
    block = Filter(**config)
    assert block.create("flt", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
    outs = []
    import torch
    for x in cycles:
        inp.data.copy_(torch.from_numpy(x))
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
        outs.append(block.output("buffer").numpy().copy())
    attrs = dict(block.output("buffer").attributes)
    block.destroy()
    return outs, attrs


@pytest.mark.parametrize("shape,taps,sr,bw", [
    ((8, 4096), 129, 8e6, 1e6),      # decimate by 8 (SURVEY.md probe: [8,4096] -> [8,1,512])
    ((8, 4096), 127, 8e6, 1e6),      # BASELINE config 3 as worded: 126 % 8 != 0 -> the reference runs at full rate
    ((4, 1024), 101, 2e6, 1e6),      # ratio 2, (taps-1) % 2 == 0, (T+taps-1) % 2 == 0 -> decimate by 2
    ((16, 512), 33, 4e6, 1e6),       # decimate by 4
    ((2048,), 65, 2e6, 2e6),         # rank 1, R = 1
    ((4, 1000), 41, 10e6, 250e3),    # R = 40
])
def test_filter_block_matches_reference_across_cycles(ref, shape, taps, sr, bw):
    from cyberether_b200.synthetic import gaussian_cf32
    config = {"sampleRate": sr, "bandwidth": bw, "taps": taps, "heads": 1}
    cycles = [gaussian_cf32(shape, 40 + i) for i in range(3)]
    want, info = _ref_filter(ref, cycles, config)
    got, attrs = _our_filter(cycles, config)
    for c, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape, (g.shape, w.shape)
        err = np.abs(w.diff(g)).max() / w.absmax()
        assert err <= 1e-5, (c, err)       # north-star tolerance, normwise per cycle
    assert attrs["sampleAxis"] == info["sample_axis"] and attrs["channelAxis"] == info["channel_axis"]
    assert attrs.get("batchAxis", -1) == info["batch_axis"]


def test_filter_taps_bit_exact(ref):
    import cyberether_b200 as cb
    ctx = cb.TestContext("filter_taps")
    ctx.set_config(sampleRate=8e6, bandwidth=1e6, center=(0.0, 1.5e6, -2e6), taps=129)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    got = ctx.output("coeffs")
    with ref.Session() as s:
        s.add_block("t", "filter_taps", {"sampleRate": 8e6, "bandwidth": 1e6, "center": [0.0, 1.5e6, -2e6], "taps": 129, "heads": 3})
        s.compute()
        want = s.output("t", "coeffs")
    assert want.equals(got)


def test_filter_multi_head_full_rate(ref):
    """Three heads with non-zero centres, no resampling (ratio not an integer): complex band-pass taps."""
    from cyberether_b200.synthetic import gaussian_cf32
    config = {"sampleRate": 3e6, "bandwidth": 1.3e6, "taps": 51, "heads": 3, "center": [0.0, 5e5, -7e5]}
    cycles = [gaussian_cf32((4, 512), 70 + i) for i in range(2)]
    want, _ = _ref_filter(ref, cycles, config)
    got, _ = _our_filter(cycles, config)
    for g, w in zip(got, want):
        assert g.shape == w.shape == (4, 3, 512)
        assert np.abs(w.diff(g)).max() / w.absmax() <= 1e-5


def test_filter_large_roundtrip_property():
    """Size-independent property at BASELINE config-3 scale (2^22 samples here): filtering a stream in one call
    equals filtering it in two calls (state carry), bit for bit."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import Filter
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((512, 8192), 9)
    def run(parts):
        block = None
        outs = []
        for part in parts:
            if block is None:
                inp = cb.Tensor.from_numpy(part, sampleAxis=1, batchAxis=0)
                block = Filter(sampleRate=8e6, bandwidth=1e6, taps=129)
                assert block.create("f", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
            else:
                inp.data.copy_(torch.from_numpy(part))
            assert block.compute() == cb.Result.SUCCESS
            outs.append(block.output("buffer").numpy().copy())
        block.destroy()
        return np.concatenate(outs, axis=0)
    whole = run([x])
    halves = run([x[:256], x[256:]])
    assert np.array_equal(whole, halves)


def _ref_fm(ref, cycles, config, axes):
    outs = []
    with ref.Session() as s:
        s.add_source("src", cycles[0], *axes)
        s.add_block("fm", "fm", config, {"signal": "src.signal"})
        for x in cycles:
            s.write_source("src", x)
            s.compute()
            outs.append(s.output("fm", "signal"))
    return outs


def _our_fm(cycles, config, axes):
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import FmBlock
    names = dict(zip(("sampleAxis", "batchAxis", "channelAxis"), [a if a >= 0 else None for a in axes]))
    inp = cb.Tensor.from_numpy(cycles[0], **names)
    block = FmBlock(**config)
    assert block.create("fm", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
    outs = []
    for x in cycles:
        inp.data.copy_(torch.from_numpy(x))
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
        outs.append(block.output("signal").numpy().copy())
    block.destroy()
    return outs


def _fm_signal(shape, seed, rate):
    rng = np.random.Generator(np.random.PCG64(seed))
    n = int(np.prod(shape))
    t = np.arange(n) / rate
    phase = 2 * np.pi * 20e3 / (2 * np.pi * 1e3) * np.sin(2 * np.pi * 1e3 * t)
    x = np.exp(1j * phase) + 0.01 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64).reshape(shape)


@pytest.mark.parametrize("shape,axes", [((4096,), (0, -1, -1)), ((8, 2048), (1, 0, -1)), ((4, 3, 512), (2, 0, 1))])
@pytest.mark.parametrize("deemphasis", ["none", "75us"])
def test_fm_narrow_matches_reference(ref, shape, axes, deemphasis):
    config = {"mode": "narrow", "deemphasis": deemphasis, "sampleRate": 250e3}
    cycles = [_fm_signal(shape, 5 + i, 250e3) for i in range(3)]
    cycles[1].reshape(-1)[7] = np.nan + 0j          # non-finite samples emit NaN without poisoning state
    want = _ref_fm(ref, cycles, config, axes)
    got = _our_fm(cycles, config, axes)
    for g, w in zip(got, want):
        assert g.shape == w.shape
        assert w.same_nan(g)
        g, w = w.take(g), w.values
        m = ~np.isnan(w)
        # atan2f (CUDA vs glibc) <= 2 ulp; de-emphasis carries are re-associated: 1e-5 (reference test: 1e-5)
        assert np.abs(g[m] - w[m]).max() <= 1e-5


@pytest.mark.parametrize("shape,axes", [((64, 8192), (1, 0, -1)), ((24, 5, 4096), (2, 0, 1)), ((7, 1001), (1, 0, -1)),
                                        ((3, 2, 6150), (2, 0, 1))])
@pytest.mark.parametrize("deemphasis", ["none", "75us"])
def test_fm_narrow_many_tiles(ref, shape, axes, deemphasis):
    """The one-pass kernel's decoupled look-back over hundreds of tiles per lane, several lanes, frame lengths that are
    not a multiple of the tile or of the vector width, state carried over three cycles."""
    config = {"mode": "narrow", "deemphasis": deemphasis, "sampleRate": 250e3}
    cycles = [_fm_signal(shape, 50 + i, 250e3) for i in range(3)]
    cycles[1].reshape(-1)[4099] = np.nan + 0j
    cycles[2].reshape(-1)[0] = np.inf + 0j
    want = _ref_fm(ref, cycles, config, axes)
    got = _our_fm(cycles, config, axes)
    for g, w in zip(got, want):
        assert g.shape == w.shape
        assert w.same_nan(g)
        g, w = w.take(g), w.values
        m = ~np.isnan(w)
        assert np.abs(g[m] - w[m]).max() <= 1e-5


def test_fm_first_sample_is_zero_and_known_tone():
    """fm/module_tests.cc: out[0] of the very first sample is 0; a constant-frequency tone demodulates to a constant."""
    import cyberether_b200 as cb
    rate, f = 240e3, 10e3
    x = np.exp(2j * np.pi * f * np.arange(4096) / rate).astype(np.complex64)
    ctx = cb.TestContext("fm")
    ctx.set_input("signal", x, sampleAxis=0)
    ctx.set_config(mode="narrow", deemphasis="none", sampleRate=rate)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    out = ctx.output("signal")
    assert out[0] == 0.0
    expected = (2 * np.pi * f / rate) / (2 * np.pi * (100e3 / rate))
    assert np.abs(out[1:] - expected).max() < 1e-4


def _stereo_mpx(n, seed, rate):
    """Composite stereo multiplex (L+R, 19 kHz pilot, (L-R) DSB-SC at 38 kHz) frequency-modulated, +-75 kHz."""
    rng = np.random.Generator(np.random.PCG64(seed))
    t = (np.arange(n) + seed * n) / rate
    left, right = np.sin(2 * np.pi * 1e3 * t), 0.5 * np.sin(2 * np.pi * 3e3 * t)
    mpx = 0.45 * (left + right) + 0.1 * np.sin(2 * np.pi * 19e3 * t) + 0.45 * (left - right) * np.sin(2 * np.pi * 38e3 * t)
    phase = 2 * np.pi * 75e3 * np.cumsum(mpx) / rate
    x = np.exp(1j * phase) + 0.002 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64)


@pytest.mark.parametrize("deemphasis", ["none", "50us"])
@pytest.mark.parametrize("shape,axes", [((8, 2000), (1, 0, -1)), ((6000,), (0, -1, -1))])
def test_fm_wide_stereo_matches_reference(ref, shape, axes, deemphasis):
    """Wideband mode: pilot NCO (F32 running phase), pilot recovery, notch + low-pass biquads, stereo matrix,
    state carried across three cycles; one cycle carries a NaN sample (emits NaN, leaves filter state untouched)."""
    rate = 250e3
    config = {"mode": "wide", "deemphasis": deemphasis, "sampleRate": rate}
    n = int(np.prod(shape))
    cycles = [_stereo_mpx(n, s, rate).reshape(shape) for s in range(3)]
    cycles[1].reshape(-1)[11] = np.nan + 0j
    want = _ref_fm(ref, cycles, config, axes)
    got = _our_fm(cycles, config, axes)
    for g, w in zip(got, want):
        assert g.shape == w.shape == tuple(shape) + (2,)
        assert w.same_nan(g)
        g, w = w.take(g), w.values
        m = ~np.isnan(w)
        assert np.abs(g[m] - w[m]).max() <= 2e-5 * max(1.0, np.abs(w[m]).max())


def test_filter_multi_head_channelizer_with_resampling(ref):
    """Three heads, two with non-zero centres, decimate by 4: the reference shifts each head to baseband by
    offsetting the spectral fold (fold channelOffsets) and keeps frames phase-continuous with phase_correction,
    carried across cycles — the "multi-fm" flowgraph structure (examples/flowgraphs/multi-fm.yml)."""
    from cyberether_b200.synthetic import gaussian_cf32
    config = {"sampleRate": 4e6, "bandwidth": 1e6, "taps": 33, "heads": 3, "center": [0.0, 1e6, -1.25e6]}
    cycles = [gaussian_cf32((6, 1024), 90 + i) for i in range(3)]
    want, info = _ref_filter(ref, cycles, config)
    got, attrs = _our_filter(cycles, config)
    for c, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape == (6, 3, 256)
        err = np.abs(w.diff(g)).max() / w.absmax()
        assert err <= 1e-5, (c, err)


@pytest.mark.parametrize("deemphasis", ["none", "75us"])
def test_fm_narrow_large_split_property(deemphasis):
    """Size-independent property at 2^23 samples (4096 tiles per lane in the look-back scan): demodulating a stream in
    one call equals demodulating it in two calls with the state carried in the plan — bit for bit without de-emphasis,
    to 2e-6 with it (the carry reaches a tile through differently grouped map compositions)."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import FmBlock
    frames, fl = 1024, 8192
    x = _fm_signal((frames, fl), 77, 250e3)

    def run(parts):
        inp = cb.Tensor.from_numpy(parts[0], sampleAxis=1, batchAxis=0)
        block = FmBlock(mode="narrow", deemphasis=deemphasis, sampleRate=250e3)
        assert block.create("fm", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
        outs = []
        for part in parts:
            inp.data.copy_(torch.from_numpy(part))
            assert block.compute() == cb.Result.SUCCESS, cb.last_error()
            outs.append(block.output("signal").numpy().copy())
        block.destroy()
        return np.concatenate(outs, axis=0)

    whole = run([x])
    halves = run([x[:512], x[512:]])
    assert whole.shape == halves.shape == (frames, fl)
    if deemphasis == "none":
        assert np.array_equal(whole, halves)
    else:
        assert np.abs(whole - halves).max() <= 2e-6


@pytest.mark.parametrize("config", [dict(sampleRate=8e6, bandwidth=1e6, taps=129),
                                    dict(sampleRate=1e6, bandwidth=100e3, taps=101, heads=3,
                                         center=(-250e3, 0.0, 125e3))])
def test_filter_time_sharding_with_halo(config):
    """Time sharding (SURVEY.md §8e): the second half of a stream filtered by a FRESH plan whose history is the halo —
    the last taps-1 samples of the first half, what `sharding.exchange_fir_halo` delivers to the next rank — equals the
    second half of the whole-stream result bit for bit, including translating multi-head plans (frames_before)."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import Filter
    from cyberether_b200.sharding import exchange_fir_halo
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((8, 2000) if "heads" in config else (64, 8192), 21)
    split = x.shape[0] // 2

    def block_for(part):
        inp = cb.Tensor.from_numpy(part, sampleAxis=1, batchAxis=0)
        block = Filter(**config)
        assert block.create("f", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
        return block, inp

    whole_block, _ = block_for(x)
    assert whole_block.compute() == cb.Result.SUCCESS, cb.last_error()
    whole = whole_block.output("buffer").numpy().copy()
    whole_block.destroy()

    first_block, first_in = block_for(x[:split])
    assert first_block.compute() == cb.Result.SUCCESS
    first = first_block.output("buffer").numpy().copy()
    halo = exchange_fir_halo(first_in.data, config["taps"]).own_tail       # what rank 0 would send to rank 1
    first_block.destroy()

    second_block, _ = block_for(x[split:])
    assert second_block.modules["fir"].set_history(halo, frames_before=split) == cb.Result.SUCCESS, cb.last_error()
    assert second_block.compute() == cb.Result.SUCCESS
    second = second_block.output("buffer").numpy().copy()
    second_block.destroy()

    assert np.array_equal(first, whole[:split])
    if "heads" in config:
        # the frame phasor of a translating head is exp(j (phase0 + inc frame)): starting from remainder(inc * split)
        # instead of 0 changes the F64 angle by a multiple of 2 pi up to rounding
        assert np.abs(second - whole[split:]).max() <= 1e-6 * np.abs(whole).max()
    else:
        assert np.array_equal(second, whole[split:])
