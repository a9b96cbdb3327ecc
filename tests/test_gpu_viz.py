"""SURVEY.md §8 f1 — the consumers right after the spectral chain: `lineplot` (batch sum with decimation -> normalise ->
clamp -> EMA) and `waterfall` (newest rows into a ring) on this provider vs the reference modules' own computeSubmit()
(oracle/_ref: lineplot/module_impl_native_cpu.cc, waterfall/module_impl_native_cpu.cc run unmodified), and the fused
spectrum_engine -> lineplot path where the chain kernel's epilogue delivers the batch sums."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _lineplot(cycles, config, axes):
    import cyberether_b200 as cb
    from cyberether_b200.blocks import LineplotBlock
    import torch
    inp = cb.Tensor.from_numpy(cycles[0], **axes)
    block = LineplotBlock(**config)
    assert block.create("lp", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
    outs = []
    for x in cycles:
        inp.data.copy_(torch.from_numpy(x))
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
        outs.append(block.signal_points().copy())
    block.destroy()
    return outs


def _ref_lineplot(ref, cycles, config, axes):
    kw = {"sample_axis": axes.get("sampleAxis", -1), "batch_axis": axes.get("batchAxis", -1),
          "channel_axis": axes.get("channelAxis", -1)}
    outs = []
    with ref.VizSession("lineplot", cycles[0].shape, config, **kw) as v:
        for x in cycles:
            v.compute(x)
            outs.append(v.read(select=lambda a: a.reshape(-1, 2)))
    return outs


@pytest.mark.parametrize("shape,config,axes", [
    ((64, 4096), {}, {"sampleAxis": 1, "batchAxis": 0}),
    ((64, 4096), {"decimation": 4, "averaging": 8}, {"sampleAxis": 1, "batchAxis": 0}),
    ((7, 1000), {"decimation": 3, "averaging": 2}, {"sampleAxis": 1, "batchAxis": 0}),
    ((5, 1001), {"decimation": 2}, {"channelAxis": 1, "batchAxis": 0}),
    ((256,), {"averaging": 4}, {"sampleAxis": 0}),
    ((300, 8), {"averaging": 3}, {"sampleAxis": 0, "batchAxis": 1}),          # batch-trailing layout (strided gather)
])
def test_lineplot_small_batches_bit_exact(ref, shape, config, axes):
    """Up to 64 rows one CTA column sums in the reference's own order: identical signalPoints over four cycles,
    including the EMA state carried between them."""
    rng = np.random.default_rng(11)
    cycles = [rng.uniform(0.0, 1.3, shape).astype(np.float32) for _ in range(4)]
    got = _lineplot(cycles, config, axes)
    want = _ref_lineplot(ref, cycles, config, axes)
    for g, w in zip(got, want):
        assert w.equals(g)
    if axes == {"sampleAxis": 1, "batchAxis": 0}:
        # the whole output: the restatement pinned to the reference (batch-leading layout)
        from oracle import port
        p = port.Lineplot(shape[1], batches=shape[0], decimation=config.get("decimation", 1),
                          averaging=config.get("averaging", 1))
        for g, x in zip(got, cycles):
            assert np.array_equal(g, p.compute(x))


def test_lineplot_nonfinite_input_is_clamped(ref):
    """lineplot/module_tests.cc:363-425: -inf spectra (zero-power bins in dB) stay finite after the clamp."""
    cycles = [np.full((2, 4), -np.inf, np.float32), np.ones((2, 4), np.float32), np.full((2, 4), 2.0, np.float32)]
    got = _lineplot(cycles, {"averaging": 2}, {"sampleAxis": 1, "batchAxis": 0})
    want = _ref_lineplot(ref, cycles, {"averaging": 2}, {"sampleAxis": 1, "batchAxis": 0})
    for g, w in zip(got, want):
        assert np.all(np.isfinite(g)) and np.array_equal(g, w.array())


@pytest.mark.parametrize("shape,config", [((1000, 4096), {}), ((4096, 1024), {"decimation": 2, "averaging": 5}),
                                           ((777, 333), {"decimation": 3})])
def test_lineplot_large_batches_within_reassociation_tolerance(ref, shape, config):
    """More than 64 rows: the batch sum is split over CTAs and reduced in a fixed order — a reassociation of the
    reference's sequential F32 sum. Bound: a sum of B values in [0, 1.3] carries at most ~B * eps relative error in
    either order; after normalisation (2 / B) the amplitude differs by <= 4 eps * 1.3 * sqrt(B)-ish. Asserted: 2e-6
    absolute on amplitudes in [-1, 1] (north-star tolerance 1e-5), and bit-identical run to run."""
    rng = np.random.default_rng(5)
    cycles = [rng.uniform(0.0, 1.0, shape).astype(np.float32) for _ in range(3)]
    axes = {"sampleAxis": 1, "batchAxis": 0}
    got = _lineplot(cycles, config, axes)
    again = _lineplot(cycles, config, axes)
    want = _ref_lineplot(ref, cycles, config, axes)
    for g, a, w in zip(got, again, want):
        assert np.array_equal(g, a)
        column = w.idx % 2
        assert np.array_equal(w.take(g)[column == 0], w.values[column == 0])
        assert np.abs(w.diff(g)[column == 1]).max() <= 2e-6


@pytest.mark.parametrize("batches,height,n", [(1, 5, 3), (5, 5, 3), (6, 5, 3), (13, 5, 8), (3, 5, 8), (700, 512, 4096),
                                              (100, 512, 1000)])
def test_waterfall_ring_matches_reference(ref, batches, height, n):
    import cyberether_b200 as cb
    from cyberether_b200.blocks import WaterfallBlock
    import torch
    from oracle import port
    expected = port.Waterfall(n, height)              # the whole ring: the restatement pinned to the reference
    rng = np.random.default_rng(2)
    cycles = [rng.standard_normal((batches, n)).astype(np.float32) for _ in range(4)]
    inp = cb.Tensor.from_numpy(cycles[0], sampleAxis=1, batchAxis=0)
    block = WaterfallBlock(height=height)
    assert block.create("wf", {"signal": inp}) == cb.Result.SUCCESS, cb.last_error()
    with ref.VizSession("waterfall", (batches, n), {"height": height}, sample_axis=1, batch_axis=0) as v:
        for x in cycles:
            inp.data.copy_(torch.from_numpy(x))
            assert block.compute() == cb.Result.SUCCESS, cb.last_error()
            v.compute(x)
            assert v.read(select=lambda a: a.reshape(height, n)).equals(block.frequency_bins())
            assert block.write_index == v.write_index()
            assert np.array_equal(block.frequency_bins(), expected.compute(x)) and block.write_index == expected.write_index
    block.destroy()


def test_waterfall_batch_trailing_layout(ref):
    """waterfall/module_tests.cc:542-600: [3, 2] with sampleAxis 0 / batchAxis 1 == [2, 3] batch-leading."""
    import cyberether_b200 as cb
    from cyberether_b200.blocks import WaterfallBlock
    lead = np.array([[1, 2, 3], [4, 5, 6]], np.float32)
    outs = []
    for arr, axes in ((lead, {"sampleAxis": 1, "batchAxis": 0}), (np.ascontiguousarray(lead.T), {"sampleAxis": 0, "batchAxis": 1}),
                      (lead, {"channelAxis": 1, "batchAxis": 0})):
        block = WaterfallBlock(height=4)
        assert block.create("wf", {"signal": cb.Tensor.from_numpy(arr, **axes)}) == cb.Result.SUCCESS, cb.last_error()
        assert block.compute() == cb.Result.SUCCESS
        outs.append(block.frequency_bins().copy())
        block.destroy()
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])
    assert np.array_equal(outs[0][:2], lead)


@pytest.mark.parametrize("rows,scale,dtype", [(48, True, "CF32"), (700, True, "CF32"), (700, False, "CF32"), (300, True, "CI8")])
def test_fused_chain_column_sums_feed_the_lineplot(ref, rows, scale, dtype):
    """spectrum_engine(publishColumnSums) -> lineplot: the chain kernel's epilogue accumulates the batch sums
    (b200_chain_exec_colsum), the lineplot module never reads the [rows, 4096] spectra. Checked against (a) the same
    lineplot module fed the same spectra WITHOUT the attribute (row-split kernel) and (b) the reference
    spectrum_engine -> lineplot on the CPU."""
    import torch
    import cyberether_b200 as cb
    from cyberether_b200.blocks import LineplotBlock, SpectrumEngine
    from cyberether_b200.jetstream import SpectralChain, SynchronousScheduler
    from cyberether_b200.synthetic import spectral_rows
    cycles = [spectral_rows(31 * k, rows) for k in range(3)]
    if dtype == "CI8":
        cycles = [np.stack([np.clip(np.round(c.real * 127), -128, 127), np.clip(np.round(c.imag * 127), -128, 127)],
                           axis=-1).astype(np.int8) for c in cycles]
    cfg = {"averaging": 3, "decimation": 2}
    sched = SynchronousScheduler()
    if dtype == "CI8":
        from cyberether_b200.jetstream import build_module, TensorLink
        inp = cb.Tensor.from_numpy(cycles[0], dtype="CI8", sampleAxis=1, batchAxis=0)
        chain_block = None
        win = build_module("window"); assert win.create("w", {"size": 4096}, {}) == cb.Result.SUCCESS
        inv = build_module("invert"); assert inv.create("i", None, {"signal": win.outputs["window"]}) == cb.Result.SUCCESS
        chain = build_module("spectral_chain")
        assert chain.create("c", {"enableScale": scale, "publishColumnSums": True},
                            {"buffer": TensorLink(tensor=inp), "window": inv.outputs["signal"]}) == cb.Result.SUCCESS, cb.last_error()
        for m in (win, inv, chain):
            assert sched.add(m) == cb.Result.SUCCESS
        spectra_link = chain.outputs["buffer"]
    else:
        inp = cb.Tensor.from_numpy(cycles[0], sampleAxis=1, batchAxis=0)
        chain_block = SpectrumEngine(enableScale=scale, publishColumnSums=True)
        assert chain_block.create("spec", {"buffer": inp}, scheduler=sched) == cb.Result.SUCCESS, cb.last_error()
        spectra_link = chain_block.outputs["buffer"]
    assert isinstance(spectra_link.tensor.attributes.get(SpectralChain.COLUMN_SUMS_ATTRIBUTE), cb.Tensor)
    fused = LineplotBlock(**cfg)
    assert fused.create("lp", {"signal": spectra_link}, scheduler=sched) == cb.Result.SUCCESS, cb.last_error()
    assert fused.modules["lineplot"]._colsum is not None
    plain_in = cb.Tensor.from_numpy(np.zeros((rows, 4096), np.float32), sampleAxis=1, batchAxis=0)
    plain = LineplotBlock(**cfg)
    assert plain.create("lp2", {"signal": plain_in}) == cb.Result.SUCCESS
    assert plain.modules["lineplot"]._colsum is None
    ref_lp = ref.VizSession("lineplot", (rows, 4096), cfg, sample_axis=1, batch_axis=0)
    for x in cycles:
        inp.data.copy_(torch.from_numpy(x))
        assert sched.compute() == cb.Result.SUCCESS, cb.last_error()
        spectra = spectra_link.tensor.numpy()
        plain_in.data.copy_(torch.from_numpy(spectra))
        assert plain.compute() == cb.Result.SUCCESS
        g, p = fused.signal_points(), plain.signal_points()
        # (a) same spectra, two summation orders
        assert np.abs(g[:, 1] - p[:, 1]).max() <= 2e-6 and np.array_equal(g[:, 0], p[:, 0])
        # (b) the reference chain + reference lineplot on the CPU (CF32 only; the reference has no fused integer ingest)
        if dtype == "CF32":
            want_spectra = ref.spectrum_engine(x, enable_scale=scale)
            ref_lp.compute(want_spectra)
            w = ref_lp.read(select=lambda a: a.reshape(-1, 2))
            # spectra differ within the chain allowance (noise-floor bins up to ~0.2 dB); averaged over `rows` and
            # mapped to [-1, 1]: dB outputs are clamped at -1 (all far below 0), range outputs compared at 2e-4
            assert np.abs(w.diff(g)[w.idx % 2 == 1]).max() <= (2e-4 if scale else 1e-6)
    ref_lp.close()
    fused.destroy()
    plain.destroy()
