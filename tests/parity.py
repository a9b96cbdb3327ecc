"""Parity tolerances for the spectral chain (test infrastructure).

north_star: "output within 1e-5 relative of the reference". For the complex spectrum that is a normwise
statement: max|a-b| <= 1e-5 * max|b| per transform (SURVEY.md §7 "Tolerance definition"). The dB and range
outputs are nonlinear in the spectrum, so the same statement is propagated through d(dB)/d|X| = 8.686/|X|:
a bin at level |X_k| may move by 8.686 * delta * max|X| / |X_k| dB. Both FP32 FFTs (pocketfft and ours)
sit at delta ~ 2e-7 (measured: the reference itself deviates from the F64 truth by up to 0.2 dB on
noise-floor bins); the tests use DELTA = 1e-6, ten times tighter than the north-star figure.

On top of that Backend::ApproxLog10 (helpers.hh:61-74) is discontinuous by 0.0021 dB where |X| crosses a
power of two, so an element whose magnitude sits within rounding of 2^k may legitimately differ by that
step; the tests bound how many such elements there are and how far they go.
"""
import numpy as np

DELTA = 1e-6          # normwise relative spectrum perturbation allowed (north-star: 1e-5)
DB_FLOOR_TOL = 3e-4   # dB: polynomial / affine evaluation-order rounding
DB_STEP = 2.2e-3      # dB: ApproxLog10 octave discontinuity
STEP_FRACTION = 2e-3  # at most this fraction of elements may use the step allowance


def approx_log10_f64(mag):
    f, e = np.frexp(mag)
    y = ((1.23149591368684 * f - 4.11852516267426) * f + 6.02197014179219) * f - 3.13396450166353 + e
    return y * 0.3010299956639812


def true_spectrum(x, window):
    """F64 spectrum of x * window (window = the reference's own CF32 taps, sign-flipped)."""
    return np.fft.fft(x.astype(np.complex128) * window.astype(np.complex128), axis=-1)


def db_allowance(spec_f64):
    mag = np.abs(spec_f64)
    peak = mag.max(axis=-1, keepdims=True)
    with np.errstate(divide="ignore", invalid="ignore"):
        allow = 8.686 * DELTA * peak / mag + DB_FLOOR_TOL
    return np.where(mag > 0, allow, np.inf)


def _at_sample(want, *full):
    """`want` may be a stored sample of the reference output (tests/reference_outputs.py): the full arrays `full` are
    then compared at its positions only."""
    if hasattr(want, "row_absmax"):
        return (want.values,) + tuple(want.take(a) for a in full)
    return (want,) + full


def assert_db_close(got, want, spec_f64, scale=1.0, floor=0.0):
    """|got - want| within the propagated allowance (optionally mapped through a slope `scale`)."""
    if hasattr(want, "row_absmax"):
        # a stored sample holds every non-finite reference element: no other element of `got` may be non-finite
        assert int((~np.isfinite(got)).sum()) == want.nonfinite(), "non-finite count differs"
    want, got, allow = _at_sample(want, got, np.broadcast_to(db_allowance(spec_f64) * scale + floor, np.shape(got)))
    finite = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), finite), "non-finite pattern differs"
    err = np.abs(np.where(finite, got - want, 0.0))
    over = err > allow
    assert float(over.mean()) <= STEP_FRACTION, f"{over.mean():.3e} of elements beyond allowance"
    worst = (err - allow)[over].max() if over.any() else 0.0
    assert worst <= DB_STEP * scale, f"worst excess {worst:.3e}"
    return float(err.max()), float(over.mean())


# --- strong-bin statistic (VERDICT r01 "what's weak" 3) -------------------------------------------------------------
# On bins within STRONG_DB of the row maximum the normwise allowance above is at most 8.686 * DELTA * 10^(STRONG_DB/20)
# dB, so a plain absolute bound holds there. Two FP32 FFTs (pocketfft radix-4/8 and our radix-16) each carry an error
# of ~1e-7 * max|X| per bin, i.e. up to ~1e-4 relative on a bin 60 dB below the peak = 1e-3 dB; the ApproxLog10 octave
# step (2.1e-3 dB) can hit a strong bin whose magnitude sits within rounding of a power of two, so the statistic
# reports both the bulk figure and the number of step crossings.
STRONG_DB = 60.0
STRONG_DB_TOL = 1e-3          # dB, bins within 60 dB of the row maximum
STRONG_RANGE_TOL = 1e-5       # range units per 1e-3 dB * slope 2/120 = 1.7e-5; asserted as max(1e-5, slope * 1e-3)
STRONG_STEP_FRACTION = 1e-3   # strong bins that may sit on an ApproxLog10 octave step


def strong_bin_stats(got, want, spec_f64, slope=None):
    """Error statistics of `got` vs `want` (dB, or range output when `slope` = d(range)/d(dB) max) restricted to the
    bins within STRONG_DB of their row's maximum. Returns a dict; assert_strong_bins() asserts on it."""
    mag = np.abs(spec_f64)
    peak = mag.max(axis=-1, keepdims=True)
    want, got, strong = _at_sample(want, got, mag >= peak * 10.0 ** (-STRONG_DB / 20.0))
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))[strong]
    tol = STRONG_DB_TOL if slope is None else max(STRONG_RANGE_TOL, slope * STRONG_DB_TOL)
    step = DB_STEP if slope is None else DB_STEP * slope
    over = err > tol
    return {"strong_bins": int(strong.sum()), "max": float(err.max()) if err.size else 0.0,
            "p999": float(np.quantile(err, 0.999)) if err.size else 0.0, "median": float(np.median(err)) if err.size else 0.0,
            "tol": tol, "over_fraction": float(over.mean()) if err.size else 0.0,
            "worst_excess": float((err[over] - tol).max()) if over.any() else 0.0, "step": step}


def assert_strong_bins(got, want, spec_f64, slope=None, label=""):
    st = strong_bin_stats(got, want, spec_f64, slope)
    assert st["over_fraction"] <= STRONG_STEP_FRACTION, f"{label}: {st}"
    assert st["worst_excess"] <= st["step"], f"{label}: {st}"
    return st
