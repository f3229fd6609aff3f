"""CPU suite (no GPU): pins the oracle.

1. oracle FFT vs numpy/scipy (the DFT contract FFTW3 publishes);
2. the restatement vs the committed golden fixtures (outputs of the reference's own filter.c);
3. the restatement vs the reference's own slicing loops, every shift (also golden fixtures);
4. analytic known-answer tests derived from the reference code paths (SURVEY.md 8c).
"""
import hashlib
from pathlib import Path

import numpy as np
import pytest

from conftest import rel_err

GOLD = Path(__file__).resolve().parent / "golden"


def _golden_case(name):
    z = np.load(GOLD / f"{name}.npz")
    chans = [dict(olen=int(p[0]), shift=int(p[1]), low=float(p[2]), high=float(p[3]), beta=float(p[4]), isb=bool(p[5]))
             for p in z["chan_params"]]
    notch = None if (len(z["notch"]) == 1 and z["notch"][0] == -1) else [int(b) for b in z["notch"]]
    return z, chans, notch


def _golden_stream(oracle, z):
    a, n, f, s = z["sig"]
    L, nb = int(z["L"]), int(z["nb"])
    if int(z["in_type"]) == oracle.KO_REAL:
        return oracle.siggen_real(nb * L, a, n, f, s)
    return oracle.siggen_complex(nb * L, a, n, f, s)


@pytest.mark.parametrize("n", [1, 2, 3, 4, 5, 7, 12, 49, 60, 300, 600, 1200, 1250, 1296, 30000])
def test_oracle_fft_matches_numpy(oracle, n):
    import ctypes as C

    lib = oracle.lib()
    rng = np.random.default_rng(n)
    x = (rng.standard_normal(n) + 1j * rng.standard_normal(n)).astype(np.complex64)
    got = oracle.forward(x)
    ref = np.fft.fft(x.astype(np.complex128))
    assert rel_err(got, ref) < 5e-7
    if n % 2 == 0 and n > 2:
        xr = rng.standard_normal(n).astype(np.float32)
        assert rel_err(oracle.forward(xr), np.fft.rfft(xr.astype(np.float64))) < 5e-7
        assert rel_err(oracle.forward_real_f64(xr), np.fft.rfft(xr.astype(np.float64))) < 1e-13


@pytest.mark.parametrize("name", ["real_small", "complex_small", "cfg1_siggen"])
def test_restatement_matches_golden(oracle, name):
    z, chans, notch = _golden_case(name)
    x = _golden_stream(oracle, z)
    # the synthetic source is pinned bit-for-bit (sig_gen.c + gauss.c + osc.c)
    assert np.array_equal(x[:16], z["x_head"])
    assert np.sum(x.astype(np.complex128)) == z["x_sum"][0]
    outs, specs = oracle.run_stream(x, int(z["L"]), int(z["M"]), chans, notch_bins=notch, keep_spectra=True)
    st = int(z["spec_stride"])
    for b in range(int(z["nb"])):
        # error measured against the block's largest bin (the sub-sample may miss the carrier)
        assert np.abs(specs[b][::st] - z["spec_sub"][b]).max() / z["spec_absmax"][b] < 2e-6
        assert abs(np.sum(np.abs(specs[b].astype(np.complex128)) ** 2) - z["spec_energy"][b]) < 1e-6 * z["spec_energy"][b]
        for i in range(len(chans)):
            ref = z[f"out{i}"][b]
            den = max(np.abs(ref).max(), 1e-12)
            assert np.abs(outs[b][i] - ref).max() / den < 2e-6, (name, b, i)
    for i, ch in enumerate(chans):
        N = int(z["L"]) + int(z["M"]) - 1
        pts = ch["olen"] * N // int(z["L"])
        R = oracle.design_response(pts, ch["olen"], N, int(z["in_type"]) == oracle.KO_REAL, ch["low"], ch["high"], ch["beta"])
        assert rel_err(R, z[f"resp{i}"]) < 1e-6


def test_restatement_matches_reference_library(oracle):
    """Against the reference's own filter.c (tests/golden/reference_library.npz, made by make_golden.py)."""
    z, _, _ = _golden_case("reference_library")
    L, M = 4800, 1201
    x = oracle.siggen_real(5 * L, 0.2, 0.05, 0.3123, 1.0)
    assert hashlib.sha256(x.tobytes()).digest() == z["x_sha"].tobytes()   # the reference's sig_gen made the same stream
    chans = [dict(olen=48, shift=s, low=-0.3, high=0.4, beta=9.0) for s in (1874, -1874, 0, 2999, -3005, 2990, 12)]
    chans.append(dict(olen=96, shift=1870, low=-0.2, high=0.2, beta=4.0, isb=True))
    assert np.array_equal(z["chan_params"], [[c["olen"], c["shift"], c["low"], c["high"], c["beta"], c.get("isb", False)]
                                             for c in chans])
    o1, s1 = oracle.run_stream(x, L, M, chans, notch_bins=[5], keep_spectra=True)
    st = int(z["spec_stride"])
    for b in range(5):
        assert np.abs(s1[b][::st] - z["spec_sub"][b]).max() / z["spec_absmax"][b] < 1e-6
        for c in range(len(chans)):
            o2 = z[f"out{c}"][b]
            den = max(np.abs(o2).max(), 1e-9)
            assert np.abs(o1[b][c] - o2).max() / den < 1e-6


def test_slice_sweep_matches_reference_library(oracle):
    """Every integer shift, REAL and COMPLEX masters, even and odd slave sizes: the restated
    slicing equals the reference's loops entry by entry (SURVEY.md 8a probe).  tests/golden/slice_sweep.npz holds the
    reference's master spectrum, responses and, for every slice it made, the master bin behind each entry (conjugated
    or not, or none); the reference's slices are rebuilt from those exactly."""
    z = np.load(GOLD / "slice_sweep.npz")
    olens = (48, 24, 40)
    assert np.array_equal(z["olens"], olens)
    for tag, in_type, L, M in (("real", oracle.KO_REAL, 480, 121), ("complex", oracle.KO_COMPLEX, 480, 121)):
        N = L + M - 1
        X = z[f"{tag}_X"]
        lim = N // 2 if in_type == oracle.KO_COMPLEX else N
        assert len(z[f"{tag}_src0"]) == 2 * lim - 1
        for i, olen in enumerate(olens):
            R = z[f"{tag}_R{i}"]
            assert len(R) == olen * N // L
            for shift, src in zip(range(-lim + 1, lim), z[f"{tag}_src{i}"]):
                fd = oracle.rebuild_slice(X, R, src)
                mine = oracle.slice_multiply(in_type, X, R, shift)
                assert np.abs(mine - fd).max() <= 2e-7 * np.abs(fd).max() + 1e-12, (in_type, shift, i)


def test_analytic_kat_tone_gain(oracle):
    """Real tone A*cos at an exact bin centre divisible by the overlap factor: constant complex
    output of magnitude A/sqrt(2) from block 1 on (filter.c:1020-1025; SURVEY.md 8c-i)."""
    L, M = 4800, 1201
    N = L + M - 1
    b, A = 1500, 0.1
    n = np.arange(4 * L)
    x = (A * np.cos(2 * np.pi * b * n / N)).astype(np.float32)
    out, _ = oracle.run_stream(x, L, M, [dict(olen=480, shift=b, low=-0.3, high=0.3, beta=11.0)])
    for blk in (1, 2, 3):
        assert np.allclose(np.abs(out[blk][0]), A / np.sqrt(2), rtol=2e-4)
    # shift mod V != 0: raw output steps -(shift mod V)/V revolutions per block (radio.c:1491-1497)
    b2 = 1501
    x2 = (A * np.cos(2 * np.pi * b2 * n / N)).astype(np.float32)
    out2, _ = oracle.run_stream(x2, L, M, [dict(olen=480, shift=b2, low=-0.3, high=0.3, beta=11.0)])
    ph = [np.angle(out2[blk][0][0]) / (2 * np.pi) for blk in (1, 2, 3)]
    step = ((ph[1] - ph[0] + 0.5) % 1.0) - 0.5
    assert abs(step - (-0.2)) < 1e-3
    # inverted spectrum is the complex conjugate (filter.c:876)
    outn, _ = oracle.run_stream(x, L, M, [dict(olen=480, shift=-b, low=-0.3, high=0.3, beta=11.0)])
    assert np.abs(outn[2][0] - np.conj(out[2][0])).max() < 1e-6


def test_convert_i16(oracle):
    x = np.array([0, 1, -1, 32767, -32768, 32766, -32766, 3, -4], np.int16)
    f, e, c = oracle.convert_i16(x, np.float32(0.5))
    assert np.array_equal(f, x.astype(np.float32) * np.float32(0.5))
    assert e == int(np.sum(x.astype(np.int64) ** 2)) and c == 2
    f2, _, _ = oracle.convert_i16(x, np.float32(1.0), randomize=True)
    exp = np.where(x & 1, x ^ np.int16(-2), x).astype(np.float32)
    assert np.array_equal(f2, exp)


def test_zero_input_and_empty_stream(oracle):
    L, M = 480, 121
    out, _ = oracle.run_stream(np.zeros(2 * L, np.float32), L, M, [dict(olen=48, shift=10, low=-0.3, high=0.3, beta=5.0)])
    assert all(np.all(o[0] == 0) for o in out)
    out, _ = oracle.run_stream(np.zeros(0, np.float32), L, M, [dict(olen=48, shift=10, low=-0.3, high=0.3, beta=5.0)])
    assert out == []
