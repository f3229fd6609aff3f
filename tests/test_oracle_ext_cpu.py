"""CPU suite (no GPU): pins the oracle's restatement of the slice variants and of the per-channel steps after the
filter (SURVEY.md 8a REAL-out / beam rows, 8f-1 fine tuning + power, 8f-2 noise estimate) against what the reference's
OWN code, compiled unmodified, computed: filter.c (oracle/_ref/libka9qref.so) and radio.c's downconvert() with its static
estimate_noise() (oracle/_ref/libka9qradio.so).  Those outputs are stored under tests/golden by make_golden.py, long vectors
as every k-th entry plus the last few, next to the largest magnitude of the whole vector (the denominator of the relative
error), together with the parameters they were made with."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

GOLD = Path(__file__).resolve().parent / "golden"


def _rel_sub(mine, ref_sub, ref_tail, ref_absmax, stride):
    """max|mine - ref| / max|ref| over the stored entries of ref: ref_sub = ref[::stride], ref_tail = its last entries"""
    mine = np.asarray(mine)
    d = max(np.abs(mine[::stride] - ref_sub).max(), np.abs(mine[len(mine) - len(ref_tail):] - ref_tail).max())
    return float(d) / float(ref_absmax)


# ------------------------------------------------------------------ oscillator ---------------------------------
OSC_CASES = [(0.0123, 0.0), (-0.25, 0.0), (1e-3, 1e-9), (0.0, 0.0)]


@pytest.mark.parametrize("f,r", OSC_CASES)
def test_osc_restatement_vs_reference_osc(oracle, f, r):
    n = 40000  # crosses two renormalisations (osc.c:15: every 16384 steps)
    z = np.load(GOLD / "osc_samples.npz")
    assert np.array_equal(z["cases"], OSC_CASES)
    idx, ref = z["idx"], z[f"osc{OSC_CASES.index((f, r))}"]   # osc.c's values at steps idx
    st = oracle.FineTune._S()
    o = oracle.lib()
    o.ko_osc_set(C.byref(st), f, r)
    o.ko_osc_step.argtypes = [C.c_void_p]

    class _CD(C.Structure):
        _fields_ = [("re", C.c_double), ("im", C.c_double)]

    o.ko_osc_step.restype = _CD
    got = np.empty(n, np.complex128)
    for i in range(n):
        v = o.ko_osc_step(C.byref(st))
        got[i] = complex(v.re, v.im)
    assert np.abs(got[idx] - ref).max() < 1e-10  # FMA contraction differs between the two builds; 4e4 recursive products
    # closed form the GPU epilogue uses: phase_n = n f + r n (n+1) / 2 cycles
    k = idx.astype(np.float64)
    closed = np.exp(2j * np.pi * ((k * f + r * k * (k + 1) / 2) % 1.0))
    assert np.abs(closed - ref).max() < 1e-8


# ------------------------------------------------------------------ downconvert: fine tuning, power, noise ------
def _downconvert_case(oracle, name, in_type, L, M, fs, fe_freq, chans, freq_plan, nb):
    """chans: list of (olen, out_rate, low, high, beta); freq_plan[b][c] = carrier frequency for block b.
    Compared with the reference's downconvert() on the same stream: tests/golden/<name>.npz."""
    z = np.load(GOLD / f"{name}.npz")
    assert np.array_equal(z["plan"], freq_plan) and np.array_equal(z["chans"], chans)
    sst, st = int(z["spec_stride"]), int(z["stride"])
    N = L + M - 1
    if in_type == oracle.KO_REAL:
        x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.1234, 1.0)
    else:
        x = oracle.siggen_complex(nb * L, 0.1, 0.02, 0.1234, 1.0)
    resp = [oracle.design_response(c[0] * N // L, c[0], N, in_type == oracle.KO_REAL, c[2], c[3], c[4]) for c in chans]
    fts = [oracle.FineTune(L, M, c[1]) for c in chans]
    n0 = [float("nan")] * len(chans)
    worst = dict(bb=0.0, pw=0.0, n0=0.0)
    for b in range(nb):
        X = oracle.forward(oracle.block_window(x, L, M, b))
        assert _rel_sub(X, z["spec_sub"][b], z["spec_sub_tail"][b], z["spec_absmax"][b], sst) < 1e-6
        for i, c in enumerate(chans):
            # restatement: radio.c:1437-1441 -> compute_tuning -> slice/IFFT -> noise -> fine tune -> power
            freq = -(0.0 + (fe_freq - freq_plan[b][i]))
            rc, shift, rem = oracle.compute_tuning(N, fs, freq)
            assert rc == 0 and shift == z["shift"][b, i] and rem == z["remainder"][b, i]
            y = oracle.channel_block(in_type, X, resp[i], shift)[-c[0]:].copy()
            est = oracle.estimate_noise(in_type, X, len(resp[i]), shift, fs)
            n0[i] = est if np.isnan(n0[i]) else n0[i] + 0.10 * (est - n0[i])  # radio.c:1468-1474, Power_alpha
            pw = fts[i].block(y, shift, rem)
            worst["bb"] = max(worst["bb"], _rel_sub(y, z[f"bb{i}"][b], z[f"bb{i}_tail"][b], z["bb_absmax"][b, i], st))
            worst["pw"] = max(worst["pw"], abs(pw - z["bb_power"][b, i]) / z["bb_power"][b, i])
            worst["n0"] = max(worst["n0"], abs(n0[i] - z["n0"][b, i]) / z["n0"][b, i])
    return worst


def test_downconvert_real_master_vs_reference_radio(oracle):
    L, M, fs = 4800, 1201, 240e3
    chans = [(480, 24000.0, -1 / 3, 1 / 3, 11.0), (240, 12000.0, 50 / 12000, 3000 / 12000, 11.0), (960, 48000.0, -0.4, 0.4, 7.0)]
    nb = 9
    base = [30_017.3, 61_234.5, 90_000.0]  # not on bin centres: non-zero remainders, shifts not divisible by V
    plan = [list(base) for _ in range(nb)]
    for b in range(4, nb):       # retune mid-stream: shift changes -> the one-time phase term (radio.c:1494)
        plan[b][0] = 33_333.3
    for b in range(6, nb):
        plan[b][1] = 61_234.5 + 7.25  # same shift, new remainder -> set_osc only
    w = _downconvert_case(oracle, "downconvert_real", oracle.KO_REAL, L, M, fs, 0.0, chans, plan, nb)
    assert w["bb"] < 2e-6 and w["pw"] < 1e-5 and w["n0"] < 1e-5, w


def test_downconvert_complex_master_vs_reference_radio(oracle):
    L, M, fs = 4000, 1001, 200e3
    chans = [(480, 24000.0, -1 / 3, 1 / 3, 11.0), (480, 24000.0, -0.3, 0.2, 9.0)]
    nb = 7
    plan = [[10.0e6 + 23_456.7, 10.0e6 - 41_234.5] for _ in range(nb)]
    for b in range(3, nb):
        plan[b][1] = 10.0e6 - 12_000.0
    w = _downconvert_case(oracle, "downconvert_complex", oracle.KO_COMPLEX, L, M, fs, 10.0e6, chans, plan, nb)
    assert w["bb"] < 2e-6 and w["pw"] < 1e-5 and w["n0"] < 1e-5, w


def test_noise_quantile_against_numpy(oracle):
    """independent check of the order statistics inside ko_estimate_noise (numpy's linear-interpolated quantile
    is the same definition as radio.c:1761-1775)."""
    rng = np.random.default_rng(4)
    m = 30001
    X = (rng.standard_normal(m) + 1j * rng.standard_normal(m)).astype(np.complex64)
    X[7000:7100] *= 30  # a signal inside the window
    for s_bins, shift in ((600, 7050), (1200, -7050), (300, 200), (600, 29900)):
        nb = max(s_bins, 1000)
        lo = abs(shift) - nb // 2
        lo = 0 if lo < 0 else (m - nb if lo + nb > m else lo)
        e = (X[lo:lo + nb].real.astype(np.float32) ** 2 + X[lo:lo + nb].imag.astype(np.float32) ** 2).astype(np.float64)
        en = 1.5 * np.quantile(e, 0.10)
        sel = e[e <= en]
        z = 1.5 * -np.log(0.9)
        want = sel.mean() / (1 - z * np.exp(-z) / (1 - np.exp(-z))) / (m * 1e6)
        got = oracle.estimate_noise(oracle.KO_REAL, X, s_bins, shift, 1e6)
        assert abs(got - want) / want < 1e-6


# ------------------------------------------------------------------ REAL-output slaves, beam -------------------
@pytest.mark.parametrize("in_type", ["real", "complex"])
def test_realout_slaves_vs_reference_library(oracle, in_type):
    """tests/golden/realout.npz: the reference's responses and all `points` real samples of every block (whose last olen
    samples are what execute_filter_output delivers, checked when the fixture is made)."""
    z = np.load(GOLD / "realout.npz")
    st = int(z["stride"])
    it = oracle.KO_REAL if in_type == "real" else oracle.KO_COMPLEX
    L, M, nb = 4800, 1201, 3
    N = L + M - 1
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.0123, 1.0) if it == oracle.KO_REAL else oracle.siggen_complex(nb * L, 0.1, 0.02, 0.0123, 1.0)
    cases = [(480, 50 / 24000, 0.3, 11.0, 0), (960, 0.01, 0.45, 7.0, 0), (480, -0.2, 0.25, 11.0, 40), (240, 0.05, 0.3, 5.0, -7)]
    assert np.array_equal(z["cases"], cases)
    for b in range(nb):
        X = oracle.forward(oracle.block_window(x, L, M, b))
        for i, c in enumerate(cases):
            pts = c[0] * N // L
            R = oracle.design_response_realout(pts, c[0], N, it == oracle.KO_REAL, c[1], c[2], c[3])
            assert _rel_sub(R[: pts // 2 + 1], z[f"{in_type}_resp{i}"], z[f"{in_type}_resp{i}_tail"], z[f"{in_type}_resp_absmax{i}"],
                            st) < 1e-6
            mine = oracle.channel_block_realout(it, X, R, c[4])
            assert len(mine) == pts
            assert _rel_sub(mine, z[f"{in_type}_full{i}"][b], z[f"{in_type}_full{i}_tail"][b], z[f"{in_type}_full_absmax"][b, i],
                            st) < 2e-6, (b, c)


def test_beam_slaves_vs_reference_library(oracle):
    """tests/golden/beam.npz: the olen samples the reference delivered per block and slave."""
    z = np.load(GOLD / "beam.npz")
    st = int(z["stride"])
    L, M, nb = 4000, 1001, 3
    N = L + M - 1
    x = oracle.siggen_complex(nb * L, 0.1, 0.02, 0.0123, 1.0)
    cases = [(480, 615, 1.0, 0.0), (480, -615, 0.0, 1.0), (160, 300, 0.6 - 0.2j, 0.3 + 0.7j), (80, 0, 1.0, 1j), (480, 2100, 0.5, -0.5j), (480, -2150, 0.2j, 0.9)]
    assert np.array_equal(z["cases"], cases)
    # (a slice that runs into the master's Nyquist bin is left unfinished by the reference's beam loop, filter.c:775: stale memory)
    for b in range(nb):
        X = oracle.forward(oracle.block_window(x, L, M, b))
        for i, c in enumerate(cases):
            pts = c[0] * N // L
            R = oracle.design_response(pts, c[0], N, False, -0.3, 0.35, 11.0)
            mine = oracle.channel_block_beam(X, R, c[1], c[2], c[3])
            assert _rel_sub(mine[-c[0]:], z[f"dst{i}"][b], z[f"dst{i}_tail"][b], z["dst_absmax"][b, i], st) < 2e-6, (b, c)
