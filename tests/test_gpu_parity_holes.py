"""Round-2 parity holes named by VERDICT r01: (1) the BENCHMARKED FIR configuration (127 taps, R = 8) through the
C ABI directly — the block path bypasses decimation for 127 taps exactly as the reference does, so only a direct
b200_fir_* call reaches it; (2) b200_chain_exec_host (the e2e headline path) against b200_chain_exec bit for bit;
(3) the backend / memory entry points of SURVEY §8 row a14 (b200_malloc ... b200_stream_*)."""
import ctypes
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _env():
    import torch
    from cyberether_b200 import _native
    from cyberether_b200.jetstream import Context
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = _native.load()
    return torch, _native, lib, Context.get(dev), dev


def _ref_full_rate(ref, cycles, taps, select, sr=8e6, bw=1e6):
    """The reference `filter` block at FULL rate on consecutive frames (state carried by its overlap_add), each output
    cut down by `select`."""
    outs = []
    with ref.Session() as s:
        s.add_source("src", cycles[0], sample_axis=1, batch_axis=0)
        # bandwidth/sampleRate = 1/8 shapes the taps; a tap count whose (taps-1) is not a multiple of 8 makes the
        # reference bypass its resampler (block_impl.cc:64-90) -> full-rate output to subsample
        s.add_block("flt", "filter", {"sampleRate": sr, "bandwidth": bw, "taps": taps, "heads": 1}, {"signal": "src.signal"})
        for x in cycles:
            s.write_source("src", x)
            s.compute()
            outs.append(s.output("flt", "buffer", select=select))
    return outs


def _fir_direct(cycles, taps, decimation, sr=8e6, bw=1e6):
    torch, _native, lib, ctx, dev = _env()
    host_taps = np.zeros((1, taps), np.complex64)
    center = (ctypes.c_double * 1)(0.0)
    _native.check(lib.b200_filter_taps_host(sr, bw, center, 1, taps, host_taps.ctypes.data_as(ctypes.c_void_p)))
    plan = ctypes.c_void_p()
    _native.check(lib.b200_fir_plan_create(ctx.handle, host_taps.ctypes.data_as(ctypes.c_void_p), taps, 1, decimation,
                                           ctypes.byref(plan)))
    sp = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    outs = []
    for x in cycles:
        xd = torch.from_numpy(x).to(dev)
        frames, t = x.shape
        y = torch.empty(frames, 1, t // decimation, dtype=torch.complex64, device=dev)
        _native.check(lib.b200_fir_exec(plan, xd.data_ptr(), y.data_ptr(), frames, t, sp))
        torch.cuda.synchronize(dev)
        outs.append(y.cpu().numpy())
    _native.check(lib.b200_fir_plan_destroy(plan))
    return outs


@pytest.mark.parametrize("taps,shape", [(127, (8, 4096)), (127, (3, 1024)), (129, (8, 4096)), (63, (5, 512))])
def test_fir_direct_decimate_8_equals_reference_full_rate_subsampled(ref, taps, shape):
    """y[q] = y_full[8 q]: BASELINE configs[2] as worded (127 taps + decimate-by-8), three cycles with carried state."""
    from cyberether_b200.synthetic import gaussian_cf32
    cycles = [gaussian_cf32(shape, 500 + i) for i in range(3)]
    full_taps = taps if (taps - 1) % 8 else taps          # 129: the reference block would resample by itself ...
    if (taps - 1) % 8 == 0:
        # ... so for 129 taps ask the reference block for its own decimated output instead
        want = []
        with ref.Session() as s:
            s.add_source("src", cycles[0], sample_axis=1, batch_axis=0)
            s.add_block("flt", "filter", {"sampleRate": 8e6, "bandwidth": 1e6, "taps": taps, "heads": 1},
                        {"signal": "src.signal"})
            for x in cycles:
                s.write_source("src", x)
                s.compute()
                want.append(s.output("flt", "buffer"))
    else:
        want = _ref_full_rate(ref, cycles, full_taps, lambda w: w[..., ::8])
    got = _fir_direct(cycles, taps, 8)
    for c, (g, w) in enumerate(zip(got, want)):
        assert g.shape == w.shape, (g.shape, w.shape)
        err = np.abs(w.diff(g)).max() / w.absmax()
        assert err <= 1e-5, (c, err)


def test_fir_direct_127_taps_decimate_8_at_full_config3_size(ref):
    """BASELINE configs[2] at its FULL size (2^26 CF32 samples as [8192, 8192] frames) through b200_fir_*; rows
    checked against the reference: a 4-row window at three places of the stream (the reference needs the row before
    each window for its overlap state, so it runs on 5 rows and its first row is dropped)."""
    torch, _native, lib, ctx, dev = _env()
    frames, t, taps = 8192, 8192, 127
    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    x = torch.view_as_complex(torch.randn(frames, t, 2, device=dev, generator=g)).contiguous()
    host_taps = np.zeros((1, taps), np.complex64)
    center = (ctypes.c_double * 1)(0.0)
    _native.check(lib.b200_filter_taps_host(8e6, 1e6, center, 1, taps, host_taps.ctypes.data_as(ctypes.c_void_p)))
    plan = ctypes.c_void_p()
    _native.check(lib.b200_fir_plan_create(ctx.handle, host_taps.ctypes.data_as(ctypes.c_void_p), taps, 1, 8,
                                           ctypes.byref(plan)))
    sp = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    y = torch.empty(frames, 1, t // 8, dtype=torch.complex64, device=dev)
    _native.check(lib.b200_fir_exec(plan, x.data_ptr(), y.data_ptr(), frames, t, sp))
    torch.cuda.synchronize(dev)
    _native.check(lib.b200_fir_plan_destroy(plan))
    for first in (1, 4000, frames - 4):
        window = x[first - 1:first + 4].cpu().numpy()
        want = _ref_full_rate(ref, [window], taps, lambda w: w[1:, :, ::8])[0]
        got = y[first:first + 4].cpu().numpy()
        err = np.abs(want.diff(got)).max() / want.absmax()
        assert err <= 1e-5, (first, err)
    # size-independent property over the WHOLE output: DC gain of the low-pass — a constant stream settles to sum(h)
    ones = torch.ones(64, t, dtype=torch.complex64, device=dev)
    plan = ctypes.c_void_p()
    _native.check(lib.b200_fir_plan_create(ctx.handle, host_taps.ctypes.data_as(ctypes.c_void_p), taps, 1, 8,
                                           ctypes.byref(plan)))
    y1 = torch.empty(64, 1, t // 8, dtype=torch.complex64, device=dev)
    _native.check(lib.b200_fir_exec(plan, ones.data_ptr(), y1.data_ptr(), 64, t, sp))
    torch.cuda.synchronize(dev)
    _native.check(lib.b200_fir_plan_destroy(plan))
    dc = host_taps.astype(np.complex128).sum()
    assert np.abs(y1[1:].cpu().numpy() - dc).max() <= 2e-6 * abs(dc)


@pytest.mark.parametrize("rows,chunk", [(1000, 0), (1000, 256), (1000, 1000), (1000, 7), (5, 3), (4096 + 17, 1024)])
@pytest.mark.parametrize("enable_range", [1, 0])
def test_chain_exec_host_equals_chain_exec_bit_for_bit(rows, chunk, enable_range):
    """The e2e headline path (pinned host buffers, chunked 3-stream H2D / kernel / D2H pipeline) runs the same
    kernel on the same bytes as the device-resident path: outputs must be IDENTICAL, for chunk sizes that divide the
    batch, leave a ragged last chunk, exceed it, or are tiny."""
    torch, _native, lib, ctx, dev = _env()
    from cyberether_b200 import amplitude_scaling_coeff, range_coefficients
    from cyberether_b200.synthetic import spectral_rows
    n = 4096
    base = spectral_rows(0, 64)
    x_host = torch.empty(rows, n, dtype=torch.complex64, pin_memory=True)
    reps = (rows + 63) // 64
    x_host.copy_(torch.from_numpy(np.tile(base, (reps, 1))[:rows]))
    x_host[:, 7] += torch.arange(rows, dtype=torch.float32) * 1e-4          # every row distinct
    out_host = torch.zeros(rows, n, dtype=torch.float32, pin_memory=True)
    sp = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    win = torch.empty(n, dtype=torch.complex64, device=dev)
    winv = torch.empty(n, dtype=torch.complex64, device=dev)
    _native.check(lib.b200_window_blackman_cf32(ctx.handle, win.data_ptr(), n, sp))
    _native.check(lib.b200_invert_cf32(ctx.handle, win.data_ptr(), winv.data_ptr(), 1, n, 1, sp))
    torch.cuda.synchronize(dev)
    plan = ctypes.c_void_p()
    _native.check(lib.b200_chain_plan_create(ctx.handle, n, rows, winv.data_ptr(), ctypes.byref(plan)))
    coeff = amplitude_scaling_coeff(n)
    scale, offset = range_coefficients(-120.0, 0.0)
    xd = x_host.to(dev)
    out = torch.empty(rows, n, dtype=torch.float32, device=dev)
    _native.check(lib.b200_chain_exec(plan, xd.data_ptr(), out.data_ptr(), rows, coeff, enable_range, scale, offset, sp))
    torch.cuda.synchronize(dev)
    for _ in range(2):       # twice: the staging slots are reused by the second call
        out_host.zero_()
        _native.check(lib.b200_chain_exec_host(plan, x_host.data_ptr(), out_host.data_ptr(), rows, coeff, enable_range,
                                               scale, offset, chunk))
        assert torch.equal(out_host, out.cpu())
    _native.check(lib.b200_chain_plan_destroy(plan))


def test_backend_memory_and_stream_entry_points():
    """SURVEY §8 a14 / a15: b200_malloc is zero-filled like the reference's CUDA Buffer (buffer_cuda.cc:119), copies
    go through caller streams, pinned staging, stream create / synchronise / destroy."""
    torch, _native, lib, ctx, dev = _env()
    count = ctypes.c_int()
    _native.check(lib.b200_device_count(ctypes.byref(count)))
    assert count.value == torch.cuda.device_count()
    device = ctypes.c_int(-1)
    _native.check(lib.b200_ctx_device(ctx.handle, ctypes.byref(device)))
    assert device.value == dev.index
    sms = ctypes.c_int()
    _native.check(lib.b200_ctx_sm_count(ctx.handle, ctypes.byref(sms)))
    assert sms.value == torch.cuda.get_device_properties(dev).multi_processor_count
    nbytes = (1 << 20) + 13
    stream = ctypes.c_void_p()
    _native.check(lib.b200_stream_create(ctx.handle, ctypes.byref(stream)))
    d0, d1, h0, h1 = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
    _native.check(lib.b200_malloc(ctx.handle, nbytes, ctypes.byref(d0)))
    _native.check(lib.b200_malloc(ctx.handle, nbytes, ctypes.byref(d1)))
    _native.check(lib.b200_host_alloc(ctx.handle, nbytes, ctypes.byref(h0)))
    _native.check(lib.b200_host_alloc(ctx.handle, nbytes, ctypes.byref(h1)))
    a = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(h0.value))
    b = np.ctypeslib.as_array((ctypes.c_uint8 * nbytes).from_address(h1.value))
    # fresh device memory reads back as zeros
    b[:] = 0xFF
    _native.check(lib.b200_memcpy(ctx.handle, h1, d0, nbytes, 1, stream))
    _native.check(lib.b200_stream_synchronize(ctx.handle, stream))
    assert not b.any()
    # h2d -> d2d -> d2h round trip on the caller's stream
    rng = np.random.default_rng(3)
    a[:] = rng.integers(0, 256, nbytes, dtype=np.uint8)
    _native.check(lib.b200_memcpy(ctx.handle, d0, h0, nbytes, 0, stream))
    _native.check(lib.b200_memcpy(ctx.handle, d1, d0, nbytes, 2, stream))
    _native.check(lib.b200_memcpy(ctx.handle, h1, d1, nbytes, 1, stream))
    _native.check(lib.b200_stream_synchronize(ctx.handle, stream))
    assert np.array_equal(a, b)
    # memset on the stream
    _native.check(lib.b200_memset(ctx.handle, d1, 0x5A, nbytes - 5, stream))
    _native.check(lib.b200_memcpy(ctx.handle, h1, d1, nbytes, 1, stream))
    _native.check(lib.b200_stream_synchronize(ctx.handle, stream))
    assert (b[:nbytes - 5] == 0x5A).all() and np.array_equal(b[nbytes - 5:], a[nbytes - 5:])
    # zero-size and error behaviour: Result codes + message, never an exception across the boundary
    z = ctypes.c_void_p(1)
    _native.check(lib.b200_malloc(ctx.handle, 0, ctypes.byref(z)))
    assert z.value is None
    assert lib.b200_memcpy(ctx.handle, d0, h0, nbytes, 7, stream) == 1 and b"kind" in lib.b200_last_error()
    assert lib.b200_malloc(None, 16, ctypes.byref(z)) == 1
    for p in (d0, d1):
        _native.check(lib.b200_free(ctx.handle, p))
    for p in (h0, h1):
        _native.check(lib.b200_host_free(ctx.handle, p))
    _native.check(lib.b200_stream_destroy(ctx.handle, stream))


def test_strong_bin_statistic_of_the_fused_chain(ref):
    """VERDICT r01 weak-3: besides the level-dependent allowance, bins within 60 dB of their row maximum hold a plain
    absolute bound (|d dB| <= 1e-3, |d range| <= max(1e-5, slope * 1e-3)), printed and asserted."""
    import cyberether_b200 as cb
    from cyberether_b200.blocks import SpectrumEngine
    from cyberether_b200.synthetic import spectral_rows
    from oracle import port
    from parity import assert_strong_bins, true_spectrum
    x = spectral_rows(2000, 256)
    w = port.invert(port.window(4096))
    spec = true_spectrum(x, w)
    for scale in (False, True):
        block = SpectrumEngine(enableScale=scale, rangeMin=-120.0, rangeMax=0.0)
        inp = cb.Tensor.from_numpy(x, sampleAxis=1, batchAxis=0)
        assert block.create("spec", {"buffer": inp}) == cb.Result.SUCCESS, cb.last_error()
        assert block.compute() == cb.Result.SUCCESS, cb.last_error()
        got = block.output("buffer").numpy()
        block.destroy()
        want = ref.spectrum_engine(x, enable_scale=scale)
        st = assert_strong_bins(got, want, spec, slope=(2.0 / 120.0) if scale else None, label=f"scale={scale}")
        # the statistic over every bin: against the numpy restatement of the reference chain (another FP32 FFT)
        assert_strong_bins(got, port.spectrum_engine(x, enable_scale=scale), spec, slope=(2.0 / 120.0) if scale else None,
                           label=f"scale={scale} vs port")
        print(f"strong-bin statistic (within 60 dB of the row maximum), enableScale={scale}: {st}")


# ---- large power-of-two transforms: the two-pass plans (fft_tile.cuh / fft_twopass.cuh) through the C ABI ------------------

def _fft_c2c(x, forward=True, env=None, inplace=False, misalign=False):
    """b200_fft_plan_c2c + b200_fft_exec on a [batch, n] CF32 array; env = plan-creation knobs (B200_FFT_TWOPASS_*)."""
    import ctypes
    import torch
    from cyberether_b200 import _native
    from cyberether_b200.jetstream import Context
    lib = _native.load()
    dev = torch.device("cuda:0")
    ctx = Context.get(dev)
    batch, n = x.shape
    saved = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update({k: str(v) for k, v in (env or {}).items()})
    try:
        plan = ctypes.c_void_p()
        _native.check(lib.b200_fft_plan_c2c(ctx.handle, n, batch, ctypes.byref(plan)))
    finally:
        for k, v in saved.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
    if misalign:        # a view that starts on an odd sample: 8-byte but not 16-byte aligned
        base = torch.zeros(batch * n + 1, dtype=torch.complex64, device=dev)
        base[1:] = torch.from_numpy(x).to(dev).reshape(-1)
        xin = base[1:]
        assert xin.data_ptr() % 16 == 8
    else:
        xin = torch.from_numpy(x).to(dev).reshape(-1).clone()
    out = xin if inplace else torch.empty(batch * n, dtype=torch.complex64, device=dev)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _native.check(lib.b200_fft_exec(plan, xin.data_ptr(), out.data_ptr(), 1 if forward else 0, s))
    torch.cuda.synchronize()
    got = out.cpu().numpy().reshape(batch, n).copy()
    _native.check(lib.b200_fft_plan_destroy(plan))
    return got


@pytest.mark.parametrize("n", [16384, 32768, 65536, 131072])
@pytest.mark.parametrize("forward", [True, False])
def test_two_pass_fft_chunked_with_a_ragged_last_chunk(n, forward):
    """Chunk size forced down to a few transforms: 11 transforms run as several chunks with a shorter last one; tolerance
    2e-6 of the largest bin against the F64 transform (north star 1e-5; pocketfft F32 itself sits at ~3e-7)."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((11, n), 17 * n)
    chunk_mb = max(1, (4 * n * 8) >> 20)             # 4 transforms per chunk -> chunks of 4, 4, 3
    got = _fft_c2c(x, forward, env={"B200_FFT_TWOPASS_CHUNK_MB": chunk_mb})
    want = np.fft.fft(x.astype(np.complex128), axis=1) if forward else np.fft.ifft(x.astype(np.complex128), axis=1) * n
    assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max()


@pytest.mark.parametrize("n", [16384, 65536])
def test_two_pass_fft_in_place_and_misaligned_input(n):
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((5, n), 3 * n)
    want = np.fft.fft(x.astype(np.complex128), axis=1)
    scale = np.abs(want).max()
    assert np.abs(_fft_c2c(x, inplace=True) - want).max() <= 2e-6 * scale
    assert np.abs(_fft_c2c(x, misalign=True) - want).max() <= 2e-6 * scale
    assert np.abs(_fft_c2c(x, env={"B200_FFT_TWOPASS_CHUNK_MB": 1}, inplace=True) - want).max() <= 2e-6 * scale


@pytest.mark.parametrize("n", [16384, 65536])
def test_two_pass_plans_agree_with_each_other_and_with_the_four_step_plan(n):
    """Three independent decompositions of the same transform (tiled M1 x 256, radix-16 columns + rows, four-step)."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((3, n), n + 1)
    tiled = _fft_c2c(x)
    col16 = _fft_c2c(x, env={"B200_FFT_TWOPASS_TILE": 0})
    four = _fft_c2c(x, env={"B200_FFT_TWOPASS": 0})
    scale = np.abs(four).max()
    assert np.abs(tiled - four).max() <= 2e-6 * scale and np.abs(col16 - four).max() <= 2e-6 * scale


def test_fft_8192_roundtrip_and_reference(ref):
    """The 8192-point kernel's last pass takes its twiddles from one register times W_16^b constants."""
    from cyberether_b200.synthetic import gaussian_cf32
    x = gaussian_cf32((7, 8192), 99)
    got = _fft_c2c(x)
    want = ref.fft(x, forward=True)
    assert np.abs(want.diff(got)).max() <= 2e-6 * want.absmax()
    back = _fft_c2c(got, forward=False) / 8192
    assert np.abs(back - x).max() <= 1e-5 * np.abs(x).max()


@pytest.mark.parametrize("taps,decimation,heads,offset", [(127, 8, 1, 0.0), (129, 8, 3, 0.0), (41, 2, 1, 0.0), (161, 40, 1, 0.0),
                                                         (129, 8, 3, 7e5), (63, 4, 2, -1.1e6)])
def test_fir_chunk_pair_form_equals_the_sample_form(taps, decimation, heads, offset, monkeypatch):
    """fir_decim_kernel<.., PAIR> (16-byte chunks, decimation R/2, chunk-taps (h[2c], h[2c-1])) against the 8-byte form of
    the same plan over three calls with carried history: same products, a different summation order."""
    torch, _native, lib, ctx, dev = _env()
    rng = np.random.default_rng(taps)
    centers = (ctypes.c_double * heads)(*[offset * (k + 1) for k in range(heads)])     # offset != 0: complex taps
    host = np.zeros((heads, taps), np.complex64)
    _native.check(lib.b200_filter_taps_host(8e6, 8e6 / decimation / 2, centers, heads, taps, host.ctypes.data_as(ctypes.c_void_p)))
    assert (np.abs(host.imag).max() > 0) == (offset != 0.0)
    if heads > 1:
        host *= rng.uniform(0.5, 1.5, (heads, 1)).astype(np.float32)
    frames, frame_len = 6, 40 * decimation * 3
    cycles = [(rng.standard_normal((frames, frame_len)) + 1j * rng.standard_normal((frames, frame_len))).astype(np.complex64)
              for _ in range(3)]
    results = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("B200_FIR_PAIR", mode)
        plan = ctypes.c_void_p()
        _native.check(lib.b200_fir_plan_create(ctx.handle, host.ctypes.data_as(ctypes.c_void_p), taps, heads, decimation,
                                               ctypes.byref(plan)))
        s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        outs = []
        for x in cycles:
            xd = torch.from_numpy(x).to(dev)
            yd = torch.empty(frames, heads, frame_len // decimation, dtype=torch.complex64, device=dev)
            _native.check(lib.b200_fir_exec(plan, xd.data_ptr(), yd.data_ptr(), frames, frame_len, s))
            torch.cuda.synchronize()
            outs.append(yd.cpu().numpy())
        _native.check(lib.b200_fir_plan_destroy(plan))
        results[mode] = np.stack(outs)
    scale = np.abs(results["0"]).max()
    assert scale > 0 and np.abs(results["1"] - results["0"]).max() <= 2e-6 * scale


@pytest.mark.parametrize("n", [8, 12, 64, 512, 1024, 4096, 8192, 16384, 65536, 6 * 1000])
@pytest.mark.parametrize("layout", [0, 1])
def test_fft_exec_real_half_length_path(ref, n, layout):
    """b200_fft_exec_real: real rows of even length 2h through one h-point complex transform on the row itself + the mirror-pair
    unpack kernel; layout 0 = pocketfft::r2c ([h + 1] CF32), layout 1 = FFTPACK half-complex ([2h] F32). h even, odd (n = 12:
    h = 6; 6000: h = 3000 -> Bluestein), tiled (65536: h = 32768) and, for 32 <= h <= 8192, fused into the transform kernel's
    epilogue (MODE_R2C: two, three and four register passes; 5 rows leave a partial last block)."""
    torch, _native, lib, ctx, dev = _env()
    rng = np.random.default_rng(n + layout)
    batch = 5
    x = rng.standard_normal((batch, n)).astype(np.float32)
    plan = ctypes.c_void_p()
    _native.check(lib.b200_fft_plan_c2c(ctx.handle, n // 2, batch, ctypes.byref(plan)))
    xd = torch.from_numpy(x).to(dev)
    out = torch.empty((batch, n // 2 + 1), dtype=torch.complex64, device=dev) if layout == 0 else \
        torch.empty((batch, n), dtype=torch.float32, device=dev)
    s = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    for _ in range(2):          # the second call reuses the plan-owned work buffer
        _native.check(lib.b200_fft_exec_real(plan, xd.data_ptr(), out.data_ptr(), layout, s))
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    spec = np.fft.rfft(x.astype(np.float64), axis=1)
    if layout == 0:
        want = spec
    else:
        want = np.empty((batch, n))
        want[:, 0] = spec[:, 0].real
        want[:, 1:n - 1:2] = spec[:, 1:n // 2].real
        want[:, 2:n - 1:2] = spec[:, 1:n // 2].imag
        want[:, n - 1] = spec[:, n // 2].real
    assert np.abs(got - want).max() <= 2e-6 * np.abs(spec).max()
    # an input that is only 4-byte aligned is refused (the caller falls back to the composed path)
    base = torch.zeros(batch * n + 1, dtype=torch.float32, device=dev)
    assert lib.b200_fft_exec_real(plan, base[1:].data_ptr(), out.data_ptr(), layout, s) != 0
    _native.check(lib.b200_fft_plan_destroy(plan))
