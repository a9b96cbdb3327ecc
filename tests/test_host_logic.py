"""Host-side mirror of the reference Module/Block/Scheduler interface: lifecycle, validation, error behaviour,
topological order and static settlement. Runs on CPU tensors (compute itself refuses without CUDA)."""
import numpy as np
import pytest

import cyberether_b200 as cb
from cyberether_b200.blocks import Filter, FmBlock, SpectrumEngine
from cyberether_b200.jetstream import Taint, TensorLink, build_module, filter_resample_plan


def tensor(shape, dtype=np.complex64, **axes):
    return cb.Tensor.from_numpy(np.zeros(shape, dtype), device="cpu", **axes)


def link(t):
    return TensorLink(tensor=t)


def test_registry_exact_four_key_lookup():
    assert cb.list_available_modules("fft") == [("fft", "cuda", "native", "b200")]
    with pytest.raises(KeyError):
        build_module("fft", "cuda", "native", "generic")
    with pytest.raises(KeyError):
        build_module("nonexistent")


def test_fft_lifecycle_and_attributes():
    m = build_module("fft")
    x = tensor((8, 1024), sampleAxis=1, batchAxis=0)
    assert m.create("fft", {"forward": True}, {"signal": link(x)}) == cb.Result.SUCCESS
    out = m.outputs["signal"].tensor
    assert out.shape == (8, 1024) and out.dtype == "CF32"
    assert out.attribute("sampleAxis") == 1 and out.attribute("batchAxis") == 0
    assert m.taint == Taint.DISCONTIGUOUS | Taint.STATELESS
    assert m.reconfigure({"forward": False}) == cb.Result.RECREATE       # fft/module_impl.cc: reconfigure -> RECREATE


def test_fft_rejects_missing_axes_and_unknown_config():
    m = build_module("fft")
    assert m.create("fft", None, {"signal": link(tensor((4, 64)))}) == cb.Result.ERROR
    assert "signal axis metadata" in cb.last_error()
    m = build_module("fft")
    assert m.create("fft", {"bogus": 1}, {"signal": link(tensor((64,)))}) == cb.Result.ERROR
    m = build_module("fft")
    assert m.create("fft", None, {}) == cb.Result.INCOMPLETE           # unconnected declared input


def test_window_is_static_and_validates_size():
    m = build_module("window")
    assert m.create("w", {"size": 0}, {}) == cb.Result.ERROR
    m = build_module("window")
    assert m.create("w", {"size": 4096}, {}) == cb.Result.SUCCESS
    assert m.taint & Taint.STATIC_OUTPUT
    assert m.outputs["window"].tensor.attribute("sampleAxis") == 0


def test_multiply_broadcast_shapes_and_errors():
    m = build_module("multiply")
    a, b = tensor((6, 1, 4), sampleAxis=2), tensor((1, 7, 1), sampleAxis=2)
    assert m.create("m", None, {"a": link(a), "b": link(b)}) == cb.Result.SUCCESS
    assert m.outputs["product"].tensor.shape == (6, 7, 4)
    m = build_module("multiply")
    assert m.create("m", None, {"a": link(tensor((4, 5), sampleAxis=1)), "b": link(tensor((4, 6), sampleAxis=1))}) \
        == cb.Result.ERROR
    assert "not broadcastable" in cb.last_error()


def test_amplitude_and_range_coefficients():
    m = build_module("amplitude")
    assert m.create("a", None, {"signal": link(tensor((4, 4096), sampleAxis=1, batchAxis=0))}) == cb.Result.SUCCESS
    assert abs(m.scaling_coeff + 72.2472) < 1e-4 and m.outputs["signal"].tensor.dtype == "F32"
    m = build_module("amplitude")
    assert m.create("a", None, {"signal": link(tensor((4, 8)))}) == cb.Result.ERROR   # no sample/channel axis
    r = build_module("range")
    x = tensor((16,), np.float32)
    assert r.create("r", {"min": -120.0, "max": 0.0}, {"signal": link(x)}) == cb.Result.SUCCESS
    assert abs(r.scale - 1 / 120) < 1e-9 and r.offset == 1.0
    assert r.reconfigure({"min": 0.0, "max": 0.0}) == cb.Result.SUCCESS and r.scale == 0.0 and r.offset == 0.5
    r = build_module("range")
    assert r.create("r", None, {"signal": link(tensor((16,)))}) == cb.Result.ERROR      # CF32 rejected


def test_cast_bypass_aliases_input():
    m = build_module("cast")
    x = tensor((32,))
    assert m.create("c", {"outputType": "CF32"}, {"buffer": link(x)}) == cb.Result.SUCCESS
    assert m.bypass and m.outputs["buffer"].tensor.data.data_ptr() == x.data.data_ptr()


def test_spectrum_engine_wiring_fused_and_unfused():
    import torch
    # the input lives where the block's input-less modules (window) allocate: the CUDA device when one is visible
    x = cb.Tensor.from_numpy(np.zeros((64, 4096), np.complex64), device="cuda" if torch.cuda.is_available() else "cpu",
                             sampleAxis=1, batchAxis=0)
    fused = SpectrumEngine(enableScale=True)
    assert fused.create("spec", {"buffer": x}) == cb.Result.SUCCESS, cb.last_error()
    assert list(fused.modules) == ["cast_input", "window", "invert", "spectral_chain"]
    out = fused.output("buffer")
    assert out.shape == (64, 4096) and out.dtype == "F32" and out.attribute("sampleAxis") == 1
    unfused = SpectrumEngine(enableScale=True, fused=False)
    assert unfused.create("spec", {"buffer": x}) == cb.Result.SUCCESS, cb.last_error()
    assert list(unfused.modules) == ["cast_input", "window", "invert", "reshape_window", "multiply", "fft",
                                     "amplitude", "range"]       # the reference's own sequence (block_impl.cc:120-217)
    order = [m.name.split(":")[1] for m in unfused.scheduler.order]
    assert order.index("window") < order.index("invert") < order.index("multiply") < order.index("fft") \
        < order.index("amplitude") < order.index("range")
    sched = unfused.scheduler
    static = {m.name.split(":")[1] for m in sched.order if sched.is_static(m)}
    assert static == {"window", "invert", "reshape_window"}     # settle after cycle 1 (block_tests.cc:103-122)
    with_agc = SpectrumEngine(enableAgc=True, fused=False)      # agc sits between fft and amplitude (block_impl.cc:186-200)
    assert with_agc.create("s", {"buffer": x}) == cb.Result.SUCCESS, cb.last_error()
    names = list(with_agc.modules)
    assert names.index("fft") < names.index("agc") < names.index("amplitude") and "spectral_chain" not in names
    assert with_agc.modules["agc"].config["tileSize"] == 4096   # one RMS tile per spectrum
    fused_agc = SpectrumEngine(enableAgc=True)                  # 4096-point spectra: the stage lives inside the fused kernel
    assert fused_agc.create("s", {"buffer": x}) == cb.Result.SUCCESS, cb.last_error()
    assert "agc" not in fused_agc.modules and fused_agc.modules["spectral_chain"].config["enableAgc"] is True
    assert SpectrumEngine().create("s", {"buffer": tensor((4, 8))}) == cb.Result.ERROR


def test_compute_without_cuda_fails_loudly():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    block = SpectrumEngine()
    assert block.create("spec", {"buffer": tensor((2, 4096), sampleAxis=1, batchAxis=0)}) == cb.Result.SUCCESS
    assert block.compute() == cb.Result.ERROR
    assert "no CPU path" in cb.last_error()


def test_filter_resampling_conditions_match_reference():
    """src/domains/dsp/filter/block_impl.cc:64-90 — integer ratio, (taps-1) % R == 0, (T+taps-1) % R == 0."""
    assert filter_resample_plan(8e6, 1e6, 129, 4096) == 8
    assert filter_resample_plan(8e6, 1e6, 127, 4096) == 1      # BASELINE config 3 as worded: silently full rate
    assert filter_resample_plan(8e6, 3e6, 129, 4096) == 1      # non-integer ratio
    assert filter_resample_plan(8e6, 1e6, 129, 4100) == 1      # (T + taps - 1) % R != 0
    f = Filter(sampleRate=8e6, bandwidth=1e6, taps=129)
    assert f.create("f", {"signal": tensor((8, 4096), sampleAxis=1, batchAxis=0)}) == cb.Result.SUCCESS
    out = f.output("buffer")
    assert out.shape == (8, 1, 512)
    assert (out.attribute("sampleAxis"), out.attribute("channelAxis"), out.attribute("batchAxis")) == (2, 1, 0)
    assert out.attribute("sampleRate") == 1e6
    assert Filter(taps=128).create("f", {"signal": tensor((8, 4096), sampleAxis=1, batchAxis=0)}) == cb.Result.ERROR
    assert "must be odd" in cb.last_error()
    assert Filter(heads=0).create("f", {"signal": tensor((8, 4096), sampleAxis=1, batchAxis=0)}) == cb.Result.ERROR


def test_fm_validation_matches_reference_messages():
    x = tensor((4, 1024), sampleAxis=1, batchAxis=0)
    assert FmBlock(mode="medium").create("fm", {"signal": x}) == cb.Result.ERROR
    assert "Mode must be 'narrow' or 'wide'" in cb.last_error()
    assert FmBlock(deemphasis="10us").create("fm", {"signal": x}) == cb.Result.ERROR
    assert FmBlock(sampleRate=30e6).create("fm", {"signal": x}) == cb.Result.ERROR
    assert FmBlock(mode="wide", sampleRate=100e3).create("fm", {"signal": x}) == cb.Result.ERROR
    ok = FmBlock(sampleRate=250e3)
    assert ok.create("fm", {"signal": x}) == cb.Result.SUCCESS
    out = ok.output("signal")
    assert out.dtype == "F32" and out.shape == (4, 1024) and out.attribute("frequency") == 0.0


def test_scheduler_detects_cycles_and_duplicates():
    from cyberether_b200.jetstream import SynchronousScheduler
    s = SynchronousScheduler("cpu")
    m = build_module("window")
    assert m.create("w", {"size": 8}, {}) == cb.Result.SUCCESS
    assert s.add(m) == cb.Result.SUCCESS
    assert s.add(m) == cb.Result.ERROR


def test_cast_validation_and_dtypes():
    """core/cast/module_tests.cc: supported pairs, bypass on matching dtype, invalid spellings, unsupported pairs."""
    for name, np_type, is_complex, out in (("I8", np.int8, False, "F32"), ("U16", np.uint16, False, "F32"),
                                           ("CI8", np.int8, True, "CF32"), ("CU32", np.uint32, True, "CF32")):
        x = cb.Tensor.from_numpy(np.zeros((3, 5, 2) if is_complex else (3, 5), np_type), device="cpu", dtype=name,
                                 sampleAxis=1)
        assert x.dtype == name and x.shape == (3, 5) and x.rank == 2 and x.size == 15
        m = build_module("cast")
        assert m.create("c", {"outputType": out}, {"buffer": link(x)}) == cb.Result.SUCCESS, cb.last_error()
        o = m.outputs["buffer"].tensor
        assert o.dtype == out and o.shape == (3, 5) and o.attribute("sampleAxis") == 1 and not m.bypass
        m = build_module("cast")
        assert m.create("c", {"outputType": name}, {"buffer": link(x)}) == cb.Result.SUCCESS
        assert m.bypass and m.outputs["buffer"].tensor.data is x.data            # alias, not a copy
    ci8 = cb.Tensor.from_numpy(np.zeros((4, 2), np.int8), device="cpu", dtype="CI8", sampleAxis=0)
    for spelling in ("", "cf32", "CF32 ", "NONE", "NOPE"):
        m = build_module("cast")
        assert m.create("c", {"outputType": spelling}, {"buffer": link(ci8)}) == cb.Result.ERROR
        assert "Invalid output type" in cb.last_error()
    m = build_module("cast")
    assert m.create("c", {"outputType": "F32"}, {"buffer": link(ci8)}) == cb.Result.ERROR      # complex int -> real
    assert "Unsupported conversion" in cb.last_error()
    with pytest.raises(TypeError):
        cb.Tensor.from_numpy(np.zeros((4, 3), np.int8), device="cpu", dtype="CI8")               # needs a trailing (re, im)


def test_agc_validation_like_reference():
    """dsp/agc/module_impl.cc:7-45."""
    x = tensor((4, 64), sampleAxis=1, batchAxis=0)
    for bad, text in ((dict(tileSize=0), "Tile size"), (dict(reference=-1.0), "Reference"), (dict(epsilon=0.0), "Epsilon"),
                      (dict(minGain=0.0), "Minimum gain"), (dict(minGain=2.0, maxGain=1.0), "Maximum gain"),
                      (dict(maxGainChange=0.99), "gain change")):
        m = build_module("agc")
        assert m.create("a", bad, {"signal": link(x)}) == cb.Result.ERROR
        assert text in cb.last_error()
    m = build_module("agc")
    assert m.create("a", None, {"signal": link(tensor((4, 64)))}) == cb.Result.ERROR     # no signal axes
    m = build_module("agc")
    assert m.create("a", {"tileSize": 16}, {"signal": link(x)}) == cb.Result.SUCCESS
    assert m.outputs["signal"].tensor.shape == (4, 64) and m.taint == Taint.STATELESS


def test_spectral_chain_accepts_integer_input_and_limits_fused_agc():
    win = tensor((4096,), sampleAxis=0)
    ci16 = cb.Tensor.from_numpy(np.zeros((3, 4096, 2), np.int16), device="cpu", dtype="CI16", sampleAxis=1, batchAxis=0)
    m = build_module("spectral_chain")
    assert m.create("s", {"enableAgc": True}, {"buffer": link(ci16), "window": link(win)}) == cb.Result.SUCCESS
    assert m.outputs["buffer"].tensor.dtype == "F32" and m.outputs["buffer"].tensor.shape == (3, 4096)
    small = tensor((3, 1024), sampleAxis=1, batchAxis=0)
    m = build_module("spectral_chain")
    assert m.create("s", {"enableAgc": True}, {"buffer": link(small), "window": link(tensor((1024,), sampleAxis=0))}) \
        == cb.Result.ERROR
    assert "4096-point" in cb.last_error()
    real = tensor((3, 4096), dtype=np.float32, sampleAxis=1, batchAxis=0)
    m = build_module("spectral_chain")
    assert m.create("s", None, {"buffer": link(real), "window": link(win)}) == cb.Result.ERROR


# ---- round 2: ADVICE r01 fixes ------------------------------------------------------------------------------------

@pytest.mark.parametrize("mtype,port,config", [("invert", "signal", None), ("agc", "signal", None),
                                                ("fm", "signal", {"mode": "narrow"})])
def test_empty_inputs_return_a_result_not_an_exception(mtype, port, config):
    """validate() must tolerate empty inputs (docs/blocks-and-modules.md:182-186); create on a size-0 tensor then
    has to return a Result (it raised AttributeError before) and compute is a no-op."""
    m = build_module(mtype)
    x = tensor((0, 64), sampleAxis=1, batchAxis=0)
    assert m.create("m", config, {port: link(x)}) == cb.Result.SUCCESS, cb.last_error()
    assert m.outputs["signal"].tensor.shape[:2] == (0, 64)
    assert m.compute_submit(None) == cb.Result.SUCCESS


def test_fir_filter_rows_without_batch_axis_are_lanes():
    """[B, T] with sampleAxis only: B independent lanes (overlap_add/module_impl_native_cpu.cc:176-198), one carried
    history per lane; with batchAxis = 0 the rows are consecutive frames of one stream."""
    coeffs = tensor((2, 33), sampleAxis=1, channelAxis=0)
    m = build_module("fir_filter")
    assert m.create("f", {"decimation": 4}, {"signal": link(tensor((6, 256), sampleAxis=1)),
                                             "coeffs": link(coeffs)}) == cb.Result.SUCCESS, cb.last_error()
    assert (m._lanes, m._frames) == (6, 1)
    out = m.outputs["buffer"].tensor
    assert out.shape == (6, 2, 64) and not out.has_attribute("batchAxis")
    assert out.attribute("channelAxis") == 1 and out.attribute("sampleAxis") == 2
    m = build_module("fir_filter")
    assert m.create("f", {"decimation": 4}, {"signal": link(tensor((6, 256), sampleAxis=1, batchAxis=0)),
                                             "coeffs": link(coeffs)}) == cb.Result.SUCCESS
    assert (m._lanes, m._frames) == (1, 6)
    m = build_module("fir_filter")
    assert m.create("f", None, {"signal": link(tensor((300, 64), sampleAxis=1)),
                                "coeffs": link(coeffs)}) == cb.Result.ERROR
    assert "independent lanes" in cb.last_error()


def test_block_destroy_on_a_shared_scheduler_keeps_the_other_block_running():
    from cyberether_b200.jetstream import SynchronousScheduler
    sched = SynchronousScheduler("cpu")
    a, b = FmBlock(), FmBlock()
    x = tensor((4, 128), sampleAxis=1, batchAxis=0)
    assert a.create("a", {"signal": x}, scheduler=sched) == cb.Result.SUCCESS
    assert b.create("b", {"signal": x}, scheduler=sched) == cb.Result.SUCCESS
    assert [m.name for m in sched.order] == ["a:fm", "b:fm"]
    assert a.destroy() == cb.Result.SUCCESS
    assert [m.name for m in sched.order] == ["b:fm"] and set(sched.modules) == {"b:fm"}
    assert sched.runtime is not None and [m.name for m in sched.runtime.modules] == ["b:fm"]


def test_fir_halo_rejects_slabs_shorter_than_the_halo():
    import torch
    from cyberether_b200.sharding import exchange_fir_halo
    with pytest.raises(ValueError, match="shorter than"):
        exchange_fir_halo(torch.zeros(1, 64, dtype=torch.complex64), taps=129)
    halo = exchange_fir_halo(torch.arange(256, dtype=torch.float32).reshape(2, 128), taps=129)
    assert halo.shape == (128,) and torch.equal(halo.own_tail, torch.arange(128, 256, dtype=torch.float32))
