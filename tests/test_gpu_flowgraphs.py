"""BASELINE.json configs 4 and 5 as parity cases (configs[1] is bench.py; configs 0/2/3 are covered in
test_gpu_modules / test_gpu_filter_fm)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _fm_broadcast_iq(frames, frame_len, seed, rate=10e6):
    """1 kHz tone FM-modulated with 75 kHz deviation at +250 kHz offset, plus noise (SURVEY.md §8d C4)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    n = frames * frame_len
    t = (np.arange(n) + seed * n) / rate
    phase = 2 * np.pi * 250e3 * t + (75e3 / 1e3) * np.sin(2 * np.pi * 1e3 * t)
    x = np.exp(1j * phase) + 0.05 * (rng.standard_normal(n) + 1j * rng.standard_normal(n))
    return x.astype(np.complex64).reshape(frames, frame_len)


def test_config4_fm_broadcast_flowgraph(ref):
    """Filter(decimate 40) -> FM(narrow) -> [drop the head axis] -> Filter -> Amplitude over three cycles.
    The reference's filter refuses an input that already carries a channel axis (filter/block_impl.cc:258-262),
    so the head axis is dropped between the two stages on both sides (numpy reshape, bit-exact)."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import Filter, FmBlock
    frames, T = 16, 4000
    cyc = [_fm_broadcast_iq(frames, T, s) for s in range(3)]
    f1 = {"sampleRate": 10e6, "bandwidth": 250e3, "taps": 161, "heads": 1, "center": [0.0]}
    f2 = {"sampleRate": 250e3, "bandwidth": 125e3, "taps": 41, "heads": 1}
    fm = {"mode": "narrow", "deemphasis": "75us", "sampleRate": 250e3}

    # ---- reference: stage 1 (filter -> fm) and stage 2 (filter -> amplitude) as two flowgraphs
    want = []
    with ref.Session() as s1, ref.Session() as s2:
        s1.add_source("src", cyc[0], sample_axis=1, batch_axis=0)
        s1.add_block("f1", "filter", f1, {"signal": "src.signal"})
        s1.add_block("fm", "fm", fm, {"signal": "f1.buffer"})
        mid_shape = None
        for i, x in enumerate(cyc):
            s1.write_source("src", x)
            s1.compute()
            # [frames, 1, T/40] F32 with the head axis dropped: [frames, T/40]
            mid = s1.output("fm", "signal", select=lambda a: np.ascontiguousarray(a[:, 0, :]))
            assert mid.shape == (frames, T // 40)
            if i == 0:
                s2.add_source("src", mid, sample_axis=1, batch_axis=0)
                s2.add_block("f2", "filter", f2, {"signal": "src.signal"})
                s2.add_block("amp", "amplitude", None, {"signal": "f2.buffer"})
            s2.write_source("src", mid)
            s2.compute()
            want.append((mid, s2.output("f2", "buffer"), s2.output("amp", "signal")))

    # ---- ours
    x_t = cb.Tensor.from_numpy(cyc[0], sampleAxis=1, batchAxis=0)
    b1 = Filter(**f1)
    assert b1.create("f1", {"signal": x_t}) == cb.Result.SUCCESS, cb.last_error()
    bfm = FmBlock(**fm)
    assert bfm.create("fm", {"signal": b1.output("buffer")}) == cb.Result.SUCCESS, cb.last_error()
    mid_t = cb.Tensor(bfm.output("signal").data[:, 0, :], {"sampleAxis": 1, "batchAxis": 0})   # view, head dropped
    b2 = Filter(**f2)
    assert b2.create("f2", {"signal": mid_t}) == cb.Result.SUCCESS, cb.last_error()
    amp = cb.build_module("amplitude")
    from cyberether_b200.jetstream import TensorLink, NativeCudaRuntime
    assert amp.create("amp", None, {"signal": TensorLink(tensor=b2.output("buffer"))}) == cb.Result.SUCCESS
    rt = NativeCudaRuntime("amp")
    rt.create([amp])
    for i, x in enumerate(cyc):
        x_t.data.copy_(torch.from_numpy(x))
        for blk in (b1, bfm, b2):
            assert blk.compute() == cb.Result.SUCCESS, cb.last_error()
        assert rt.compute([], set(), set()) == cb.Result.SUCCESS
        mid, filt, db = want[i]
        got_mid = bfm.output("signal").numpy()
        got_filt = b2.output("buffer").numpy()
        got_db = amp.outputs["signal"].tensor.numpy()
        # The first outputs of the stream are the decimating filter filling up from zero state: |x| ~ 1e-5 of
        # full scale there, arg() of such samples is ill-conditioned in BOTH implementations, and the
        # de-emphasis IIR (18.75-sample time constant) carries that startup difference for ~200 samples.
        skip = 3 if i == 0 else 0
        assert np.abs(mid.diff(got_mid[:, 0, :]))[mid.rows() >= skip].max() <= 2e-5      # rad-scaled audio, O(1)
        assert np.abs(filt.diff(got_filt))[filt.rows() >= skip].max() <= 1e-5 * filt.absmax()
        # strong samples of the filter output (ours, within 1e-5 normwise of the reference, as just asserted)
        strong = db.take(np.abs(got_filt) > 1e-3 * filt.absmax()) & (db.rows() >= skip)
        assert np.abs(db.diff(got_db))[strong].max() <= 5e-3                 # dB of a 1e-5-normwise-accurate signal
    for blk in (b1, bfm, b2):
        blk.destroy()


def test_config5_eight_channel_layout(ref):
    """[channels=8, batch, 4096] with channelAxis=0, batchAxis=1, sampleAxis=2: every (channel, row) is an
    independent transform; the fused kernel sees one [8*batch, 4096] slab."""
    import cyberether_b200 as cb
    from cyberether_b200.blocks import SpectrumEngine
    from cyberether_b200.synthetic import spectral_rows
    import sys, os
    sys.path.insert(0, os.path.dirname(__file__))
    from parity import assert_db_close, true_spectrum
    x = spectral_rows(500, 8 * 12).reshape(8, 12, 4096)
    want = ref.run_block("spectrum_engine", {"buffer": x}, {"enableScale": True, "rangeMin": -120.0, "rangeMax": 0.0},
                         "buffer", axes={"buffer": (2, 1, 0)})
    block = SpectrumEngine(enableScale=True)
    t = cb.Tensor.from_numpy(x, sampleAxis=2, batchAxis=1, channelAxis=0)
    assert block.create("spec", {"buffer": t}) == cb.Result.SUCCESS, cb.last_error()
    assert block.compute() == cb.Result.SUCCESS, cb.last_error()
    out = block.output("buffer")
    got = out.numpy()
    assert got.shape == want.shape == (8, 12, 4096)
    assert (out.attribute("sampleAxis"), out.attribute("batchAxis"), out.attribute("channelAxis")) == (2, 1, 0)
    from oracle import port
    w = port.invert(port.window(4096))
    assert_db_close(got, want, true_spectrum(x, w), scale=2.0 / 120.0, floor=3e-7)
    block.destroy()


def test_config0_single_1024_fft_batch1(ref):
    """BASELINE configs[0]: single 1024-pt CF32 FFT module, batch 1 (the reference's CPU-runnable plumbing case)."""
    import cyberether_b200 as cb
    x = np.exp(2j * np.pi * 5 * np.arange(1024) / 1024).astype(np.complex64)
    ctx = cb.TestContext("fft")
    ctx.set_input("signal", x, sampleAxis=0)
    ctx.set_config(forward=True)
    assert ctx.run() == cb.Result.SUCCESS, cb.last_error()
    got, want = ctx.output("signal"), ref.fft(x)
    assert abs(abs(got[5]) - 1024.0) < 1e-2
    assert np.abs(want.diff(got)).max() <= 2e-6 * want.absmax()
