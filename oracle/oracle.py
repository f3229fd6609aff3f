"""oracle/oracle.py -- ctypes front end to the two CPU checkers.

TEST INFRASTRUCTURE, NOT PRODUCT.  Only tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs may import this module; the shipped path
(ka9q_radio_b200/) never does and fails loudly when its CUDA library is missing.

  Restatement  oracle/libkaoracle.so   (chan_oracle.c; functions cite reference file:line)
  Reference    oracle/_ref/libka9qref.so  (the reference's own filter.c etc. compiled unmodified,
               driven by ref_driver.c; built by oracle/Makefile where /root/reference exists)
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
KO_COMPLEX, KO_REAL, KO_SPECTRUM = 1, 2, 3  # enum filtertype, reference src/filter.h:29-34

_c64p = np.ctypeslib.ndpointer(np.complex64, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_i16p = np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS")


def build(force: bool = False) -> None:
    """Compile the restatement when it is missing; the same make builds _ref where the reference's sources are readable."""
    if force or not (HERE / "libkaoracle.so").exists():
        subprocess.run(["make", "-C", str(HERE), "-s"], check=True)


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(HERE / "libkaoracle.so"))
        L.ko_design_response.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, _c64p]
        L.ko_forward_real.argtypes = [C.c_int, _f32p, _c64p]
        L.ko_forward_complex.argtypes = [C.c_int, _c64p, _c64p]
        L.ko_forward_real_d.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.ko_slice_multiply.argtypes = [C.c_int, C.c_int, _c64p, C.c_int, _c64p, C.c_int, C.c_int, _c64p]
        L.ko_slice_multiply.restype = None
        L.ko_channel_block.argtypes = [C.c_int, C.c_int, _c64p, C.c_int, _c64p, C.c_int, C.c_int, _c64p]
        L.ko_convert_i16.argtypes = [_f32p, _i16p, C.c_int, C.c_float, C.POINTER(C.c_uint64), C.c_int]
        L.ko_apply_notches.argtypes = [C.c_void_p, _c64p]
        L.ko_apply_notches.restype = None
        L.ko_siggen_new.restype = C.c_void_p
        L.ko_siggen_new.argtypes = [C.c_double]
        L.ko_siggen_free.argtypes = [C.c_void_p]
        L.ko_siggen_real.argtypes = [C.c_void_p, _f32p, C.c_long, C.c_double, C.c_double, C.c_double]
        L.ko_siggen_complex.argtypes = [C.c_void_p, _c64p, C.c_long, C.c_double, C.c_double, C.c_double]
        L.ko_siggen_tones_i16.argtypes = [_i16p, C.c_long, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_uint64]
        L.ko_compute_tuning.argtypes = [C.c_int, C.c_double, C.c_double, C.POINTER(C.c_int), C.POINTER(C.c_double)]
        L.ko_channel_block_beam.argtypes = [C.c_int, _c64p, C.c_int, _c64p, C.c_int] + [C.c_double] * 4 + [_c64p]
        L.ko_channel_block_realout.argtypes = [C.c_int, C.c_int, _c64p, C.c_int, _c64p, C.c_int, _f32p]
        L.ko_slice_realout.argtypes = [C.c_int, C.c_int, _c64p, C.c_int, _c64p, C.c_int, _c64p]
        L.ko_slice_realout.restype = None
        L.ko_finetune_init.argtypes = [C.c_void_p]
        L.ko_finetune_init.restype = None
        L.ko_finetune_block.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, _c64p, C.c_int]
        L.ko_finetune_block.restype = C.c_double
        L.ko_osc_set.argtypes = [C.c_void_p, C.c_double, C.c_double]
        L.ko_osc_set.restype = None
        L.ko_estimate_noise.argtypes = [C.c_int, C.c_int, _c64p, C.c_int, C.c_int, C.c_double]
        L.ko_estimate_noise.restype = C.c_double
        L.ko_fm_front.argtypes = [_c64p, C.c_int, C.c_void_p, _f32p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.ko_fm_front.restype = None
        L.ko_airspy_unpack.argtypes = [_f32p, C.c_void_p, C.c_int, C.c_float, C.POINTER(C.c_uint64)]
        _lib = L
    return _lib


# ------------------------------------------------------------------ restatement wrappers -----
def design_response(points, olen, master_points, master_real, low, high, beta) -> np.ndarray:
    out = np.empty(points, np.complex64)
    r = lib().ko_design_response(points, olen, master_points, int(bool(master_real)), low, high, beta, out)
    if r != 0:
        raise ValueError("ko_design_response rejected the parameters")
    return out


def forward(window: np.ndarray) -> np.ndarray:
    """REAL float32 window -> N/2+1 bins; complex64 window -> N bins (unnormalised, sign -1)."""
    n = len(window)
    if np.iscomplexobj(window):
        w = np.ascontiguousarray(window, np.complex64)
        out = np.empty(n, np.complex64)
        lib().ko_forward_complex(n, w, out)
    else:
        w = np.ascontiguousarray(window, np.float32)
        out = np.empty(n // 2 + 1, np.complex64)
        lib().ko_forward_real(n, w, out)
    return out


def forward_real_f64(window: np.ndarray) -> np.ndarray:
    w = np.ascontiguousarray(window, np.float64)
    out = np.empty(len(w) // 2 + 1, np.complex128)
    if lib().ko_forward_real_d(len(w), w.ctypes.data, out.ctypes.data) != 0:
        raise ValueError("even length required")
    return out


def slice_multiply(in_type, spectrum, response, shift, isb=False) -> np.ndarray:
    out = np.zeros(len(response), np.complex64)
    lib().ko_slice_multiply(in_type, len(spectrum), np.ascontiguousarray(spectrum, np.complex64), len(response),
                            np.ascontiguousarray(response, np.complex64), int(shift), int(isb), out)
    return out


def rebuild_slice(spectrum, response, src) -> np.ndarray:
    """A stored slice (tests/golden/slice_sweep.npz) back as values: entry j is spectrum[k] * response[j] for src[j] = k + 1,
    conj(spectrum[k]) * response[j] for src[j] = -(k + 1), 0 for src[j] = 0; the products exactly (complex128)."""
    k = np.abs(np.asarray(src, np.int64)) - 1
    X, R = np.asarray(spectrum, np.complex128), np.asarray(response, np.complex128)
    return np.where(src == 0, 0, np.where(src < 0, np.conj(X[k]), X[k]) * R)


def channel_block(in_type, spectrum, response, shift, isb=False) -> np.ndarray:
    """All Ns samples of the inverse transform; the user-visible part is the last olen."""
    out = np.empty(len(response), np.complex64)
    lib().ko_channel_block(in_type, len(spectrum), np.ascontiguousarray(spectrum, np.complex64), len(response),
                           np.ascontiguousarray(response, np.complex64), int(shift), int(isb), out)
    return out


def convert_i16(samples: np.ndarray, scale: float, randomize=False):
    s = np.ascontiguousarray(samples, np.int16)
    out = np.empty(len(s), np.float32)
    energy = C.c_uint64(0)
    clips = lib().ko_convert_i16(out, s, len(s), scale, C.byref(energy), int(randomize))
    return out, int(energy.value), clips


def block_window(stream: np.ndarray, L: int, M: int, b: int) -> np.ndarray:
    """Window of block b: samples [b*L-(M-1), b*L+L), zeros before the stream start."""
    start = b * L - (M - 1)
    n = L + M - 1
    out = np.zeros(n, stream.dtype)
    lo = max(start, 0)
    out[lo - start:] = stream[lo:start + n]
    return out


def siggen_real(n, amplitude, noise, cycles_per_sample, scale) -> np.ndarray:
    g = lib().ko_siggen_new(cycles_per_sample)
    out = np.empty(n, np.float32)
    lib().ko_siggen_real(g, out, n, amplitude, noise, scale)
    lib().ko_siggen_free(g)
    return out


def siggen_complex(n, amplitude, noise, cycles_per_sample, scale) -> np.ndarray:
    g = lib().ko_siggen_new(cycles_per_sample)
    out = np.empty(n, np.complex64)
    lib().ko_siggen_complex(g, out, n, amplitude, noise, scale)
    lib().ko_siggen_free(g)
    return out


def siggen_tones_i16(n, cycles_per_sample, amplitudes, noise, seed=1) -> np.ndarray:
    f = np.ascontiguousarray(cycles_per_sample, np.float64)
    a = np.ascontiguousarray(amplitudes, np.float64)
    out = np.empty(n, np.int16)
    lib().ko_siggen_tones_i16(out, n, len(f), f.ctypes.data, a.ctypes.data, noise, seed)
    return out


def compute_tuning(N, samprate, freq):
    sh, rem = C.c_int(0), C.c_double(0)
    r = lib().ko_compute_tuning(N, samprate, freq, C.byref(sh), C.byref(rem))
    return r, sh.value, rem.value


def channel_block_beam(spectrum, response, shift, i_weight=1.0, q_weight=0.0) -> np.ndarray:
    """COMPLEX master, beam == true (filter.c:756-775); weights as set_filter_weights takes them (filter.c:922-929)."""
    alpha = 0.5 * complex(i_weight) - 1j * complex(q_weight)
    beta = 0.5 * complex(i_weight) + 1j * complex(q_weight)
    out = np.empty(len(response), np.complex64)
    lib().ko_channel_block_beam(len(spectrum), np.ascontiguousarray(spectrum, np.complex64), len(response),
                                np.ascontiguousarray(response, np.complex64), int(shift),
                                alpha.real, alpha.imag, beta.real, beta.imag, out)
    return out


def channel_block_realout(in_type, spectrum, response, shift) -> np.ndarray:
    """REAL-output slave (filter.c:794-809 + c2r inverse): all `points` real samples; user part = last olen."""
    pts = len(response)
    out = np.empty(pts, np.float32)
    r = lib().ko_channel_block_realout(in_type, len(spectrum), np.ascontiguousarray(spectrum, np.complex64), pts,
                                       np.ascontiguousarray(response, np.complex64), int(shift), out)
    if r != 0:
        raise ValueError("REAL-output slaves need an even number of points")
    return out


def design_response_realout(points, olen, master_points, master_real, low, high, beta) -> np.ndarray:
    """set_filter for a REAL slave folds both edges to positive frequencies first (filter.c:971-975)."""
    return design_response(points, olen, master_points, master_real, abs(low), abs(high), beta)


def estimate_noise(in_type, spectrum, s_bins, shift, samprate) -> float:
    """radio.c:1783-1866 on one block's master spectrum."""
    return float(lib().ko_estimate_noise(in_type, len(spectrum), np.ascontiguousarray(spectrum, np.complex64),
                                         int(s_bins), int(shift), float(samprate)))


class FmFront:
    """fm.c:104-131 + :205-231 on successive blocks of one channel (phase_memory carried across blocks)"""

    def __init__(self):
        self.pm = (C.c_double * 2)(0.0, 0.0)

    def block(self, x: np.ndarray):
        x = np.ascontiguousarray(x, np.complex64)
        bb = np.empty(len(x), np.float32)
        avg, var = C.c_double(0), C.c_double(0)
        lib().ko_fm_front(x, len(x), C.cast(self.pm, C.c_void_p), bb, C.byref(avg), C.byref(var))
        return bb, avg.value, var.value


def airspy_unpack(packed_words: np.ndarray, sampcount: int, scale: float):
    """airspy-unpack.c:106-130 -> (float32[sampcount], energy, clip count)"""
    w = np.ascontiguousarray(packed_words, np.uint32)
    out = np.empty(sampcount, np.float32)
    e = C.c_uint64(0)
    over = lib().ko_airspy_unpack(out, w.ctypes.data, sampcount, scale, C.byref(e))
    return out, int(e.value), over


def airspy_pack(samples12: np.ndarray) -> np.ndarray:
    """inverse of the unpacker, for building test inputs: offset-binary 12-bit values (0..4095), 8 per 3 words"""
    s = np.asarray(samples12, np.uint64).reshape(-1, 8)
    w0 = (s[:, 0] << 20) | (s[:, 1] << 8) | (s[:, 2] >> 4)
    w1 = ((s[:, 2] & 0xF) << 28) | (s[:, 3] << 16) | (s[:, 4] << 4) | (s[:, 5] >> 8)
    w2 = ((s[:, 5] & 0xFF) << 24) | (s[:, 6] << 12) | s[:, 7]
    return np.stack([w0, w1, w2], axis=1).astype(np.uint32).reshape(-1)


class FineTune:
    """Per-channel state of radio.c:1476-1501 (fine oscillator, block phase) + :1515-1520 (power)."""

    class _S(C.Structure):
        _fields_ = [("freq", C.c_double), ("rate", C.c_double), ("phasor", C.c_double * 2), ("phasor_step", C.c_double * 2),
                    ("phasor_step_step", C.c_double * 2), ("steps", C.c_int), ("remainder", C.c_double),
                    ("bin_shift", C.c_int), ("phase_adjust", C.c_double * 2)]

    def __init__(self, L, M, out_samprate):
        self.s = self._S()
        lib().ko_finetune_init(C.byref(self.s))
        self.L, self.M, self.rate = L, M, float(out_samprate)

    def block(self, y: np.ndarray, shift: int, remainder: float, doppler_rate: float = 0.0):
        """Rotates y (complex64, olen samples) in place; returns bb_power."""
        assert y.dtype == np.complex64 and y.flags.c_contiguous
        return float(lib().ko_finetune_block(C.byref(self.s), self.L, self.M, int(shift), float(remainder), self.rate,
                                             float(doppler_rate), y, len(y)))

    @property
    def phase_cycles(self) -> float:
        """current oscillator phase in cycles"""
        return float(np.angle(complex(*self.s.phasor)) / (2 * np.pi))


class Notches:
    """Notch list (filter.c:464-474): given spur bins + implicit DC entry last."""

    class _N(C.Structure):
        _fields_ = [("bin", C.c_int), ("state", C.c_double * 2), ("alpha", C.c_double)]

    def __init__(self, bins, alpha=0.01):
        bins = list(bins) + [0]
        self.arr = (self._N * len(bins))()
        for i, b in enumerate(bins):
            self.arr[i].bin = b
            self.arr[i].alpha = alpha

    def apply(self, spectrum: np.ndarray) -> None:
        lib().ko_apply_notches(C.cast(self.arr, C.c_void_p), spectrum)


def run_stream(stream, L, M, channels, notch_bins=None, keep_spectra=False):
    """Whole restated path over a stream.

    stream: float32 (REAL master) or complex64 (COMPLEX master), length nblocks*L.
    channels: list of dicts {olen, shift, low, high, beta[, isb]}.
    Returns (outputs[nblocks][nch] -> complex64[olen], spectra or None).
    """
    in_type = KO_COMPLEX if np.iscomplexobj(stream) else KO_REAL
    N = L + M - 1
    nblocks = len(stream) // L
    resp = []
    for ch in channels:
        pts = ch["olen"] * N // L
        resp.append(design_response(pts, ch["olen"], N, in_type == KO_REAL, ch["low"], ch["high"], ch["beta"]))
    notches = Notches(notch_bins) if notch_bins is not None else None
    outs, spectra = [], []
    for b in range(nblocks):
        X = forward(block_window(stream, L, M, b))
        if notches is not None:
            notches.apply(X)
        if keep_spectra:
            spectra.append(X.copy())
        row = []
        for ch, R in zip(channels, resp):
            y = channel_block(in_type, X, R, ch["shift"], ch.get("isb", False))
            row.append(y[len(y) - ch["olen"]:].copy())
        outs.append(row)
    return outs, (spectra if keep_spectra else None)


# ------------------------------------------------------------------ the real reference -------
_ref = None


def ref_available() -> bool:
    build()
    return (HERE / "_ref/libka9qref.so").exists()


def bind_driver(R: C.CDLL) -> C.CDLL:
    """ctypes prototypes of the flat filter.h driver API (oracle/ref_driver.c, tests/abi/filter_driver.c)."""
    if True:
        R.ref_open.restype = C.c_void_p
        R.ref_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int]
        R.ref_close.argtypes = [C.c_void_p]
        R.ref_set_notches.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double]
        R.ref_add_channel.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double]
        R.ref_retune_channel.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_double]
        R.ref_channel_points.argtypes = [C.c_void_p, C.c_int]
        R.ref_get_response.argtypes = [C.c_void_p, C.c_int, _c64p]
        R.ref_set_isb.argtypes = [C.c_void_p, C.c_int, C.c_int]
        R.ref_write_real.argtypes = [C.c_void_p, _f32p, C.c_int]
        R.ref_write_complex.argtypes = [C.c_void_p, _c64p, C.c_int]
        R.ref_get_spectrum.argtypes = [C.c_void_p, _c64p]
        R.ref_master_bins.argtypes = [C.c_void_p]
        R.ref_execute_channel.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        R.ref_channel_drops.argtypes = [C.c_void_p, C.c_int]
        R.ref_channel_drops.restype = C.c_uint
    return R


def ref_lib() -> C.CDLL:
    global _ref
    if _ref is None:
        build()
        p = HERE / "_ref/libka9qref.so"
        if not p.exists():
            raise FileNotFoundError("oracle/_ref/libka9qref.so not built (needs /root/reference)")
        R = bind_driver(C.CDLL(str(p)))
        R.ref_siggen_real.argtypes = [_f32p, C.c_long, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int]
        R.ref_siggen_real.restype = None
        R.ref_siggen_complex.argtypes = [_c64p, C.c_long, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int]
        R.ref_siggen_complex.restype = None
        R.ref_bench.restype = C.c_double
        R.ref_bench.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_double,
                                C.c_double, C.c_void_p, C.c_long, C.c_int, C.c_int, C.POINTER(C.c_uint)]
        _ref = R
    return _ref


class RefSession:
    """The reference's own create_filter_input/output + execute path, inline forward FFT."""

    def __init__(self, L, M, in_type, nworkers=0, lib=None):
        self.R = lib if lib is not None else ref_lib()
        self.h = self.R.ref_open(L, M, in_type, nworkers)
        if not self.h:
            raise RuntimeError("create_filter_input failed")
        self.L, self.M, self.in_type = L, M, in_type
        self.olen = []
        self._keep = []

    def set_notches(self, bins, alpha=0.01):
        arr = (C.c_int * max(len(bins), 1))(*bins)
        self._keep.append(arr)
        self.R.ref_set_notches(self.h, C.cast(arr, C.c_void_p), len(bins), alpha)

    def add_channel(self, olen, low, high, beta, out_type=KO_COMPLEX) -> int:
        i = self.R.ref_add_channel(self.h, olen, out_type, low, high, beta)
        if i < 0:
            raise RuntimeError("create_filter_output/set_filter failed")
        self.olen.append(olen)
        return i

    def response(self, ch) -> np.ndarray:
        n = self.R.ref_channel_points(self.h, ch)
        out = np.empty(n, np.complex64)
        self.R.ref_get_response(self.h, ch, out)
        return out

    def set_isb(self, ch, isb):
        self.R.ref_set_isb(self.h, ch, int(isb))

    def write(self, samples) -> int:
        if self.in_type == KO_REAL:
            return self.R.ref_write_real(self.h, np.ascontiguousarray(samples, np.float32), len(samples))
        return self.R.ref_write_complex(self.h, np.ascontiguousarray(samples, np.complex64), len(samples))

    def spectrum(self) -> np.ndarray:
        out = np.empty(self.R.ref_master_bins(self.h), np.complex64)
        self.R.ref_get_spectrum(self.h, out)
        return out

    def execute(self, ch, shift, want_full=False, want_fdomain=False):
        n = self.R.ref_channel_points(self.h, ch)
        dst = np.empty(self.olen[ch], np.complex64)
        full = np.empty(n, np.complex64) if want_full else None
        fdom = np.empty(n, np.complex64) if want_fdomain else None
        r = self.R.ref_execute_channel(self.h, ch, int(shift), dst.ctypes.data,
                                       full.ctypes.data if want_full else None,
                                       fdom.ctypes.data if want_fdomain else None)
        if r != 0:
            raise RuntimeError("execute_filter_output returned %d" % r)
        res = [dst]
        if want_full:
            res.append(full)
        if want_fdomain:
            res.append(fdom)
        return res[0] if len(res) == 1 else tuple(res)

    def close(self):
        if self.h:
            self.R.ref_close(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def ref_run_stream(stream, L, M, channels, notch_bins=None, keep_spectra=False, lib=None):
    """Same contract as run_stream() but executed by the reference's own filter.c (or, with
    lib=<tests/abi driver>, by whatever library implements the filter.h surface)."""
    in_type = KO_COMPLEX if np.iscomplexobj(stream) else KO_REAL
    nblocks = len(stream) // L
    outs, spectra = [], []
    with RefSession(L, M, in_type, lib=lib) as s:
        if notch_bins is not None:
            s.set_notches(list(notch_bins))
        ids = [s.add_channel(ch["olen"], ch["low"], ch["high"], ch["beta"]) for ch in channels]
        for i, ch in zip(ids, channels):
            if ch.get("isb"):
                s.set_isb(i, True)
        for b in range(nblocks):
            fired = s.write(stream[b * L:(b + 1) * L])
            assert fired == 1
            if keep_spectra:
                spectra.append(s.spectrum())
            outs.append([s.execute(i, ch["shift"]) for i, ch in zip(ids, channels)])
    return outs, (spectra if keep_spectra else None)


def ref_siggen_real(n, amplitude, noise, cycles_per_sample, scale) -> np.ndarray:
    out = np.empty(n, np.float32)
    ref_lib().ref_siggen_real(out, n, amplitude, noise, cycles_per_sample, scale, 1)
    return out


def ref_siggen_complex(n, amplitude, noise, cycles_per_sample, scale) -> np.ndarray:
    out = np.empty(n, np.complex64)
    ref_lib().ref_siggen_complex(out, n, amplitude, noise, cycles_per_sample, scale, 1)
    return out


# ------------------------------------------------------------------ the reference's downconvert() --
_radio = None


def radio_available() -> bool:
    build()
    return (HERE / "_ref/libka9qradio.so").exists()


def radio_lib() -> C.CDLL:
    """oracle/_ref/libka9qradio.so: the reference's radio.c (downconvert, estimate_noise, compute_tuning) unmodified."""
    global _radio
    if _radio is None:
        build()
        p = HERE / "_ref/libka9qradio.so"
        if not p.exists():
            raise FileNotFoundError("oracle/_ref/libka9qradio.so not built (needs /root/reference)")
        R = C.CDLL(str(p))
        R.rr_open.argtypes = [C.c_int, C.c_int, C.c_int, C.c_double, C.c_double]
        R.rr_add_channel.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double]
        R.rr_set_freq.argtypes = [C.c_int, C.c_double, C.c_double, C.c_double]
        R.rr_write_real.argtypes = [_f32p, C.c_int]
        R.rr_write_complex.argtypes = [_c64p, C.c_int]
        R.rr_downconvert.argtypes = [C.c_int, _c64p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int),
                                     C.POINTER(C.c_double)]
        R.rr_get_spectrum.argtypes = [_c64p]
        R.rr_osc_run.argtypes = [C.c_double, C.c_double, C.c_long, C.c_void_p]
        R.rr_osc_run.restype = None
        R.rr_close.restype = None
        _radio = R
    return _radio


class RadioRef:
    """One front end + channels run through the reference's own downconvert() (radio.c:1410)."""

    def __init__(self, L, M, in_type, samprate, frequency=0.0):
        self.R = radio_lib()
        if self.R.rr_open(L, M, in_type, samprate, frequency) != 0:
            raise RuntimeError("rr_open failed (one session at a time)")
        self.in_type, self.olen = in_type, []

    def add_channel(self, olen, out_samprate, freq, low, high, beta) -> int:
        i = self.R.rr_add_channel(olen, out_samprate, freq, low, high, beta)
        if i < 0:
            raise RuntimeError("rr_add_channel failed")
        self.olen.append(olen)
        return i

    def set_freq(self, ch, freq, doppler=0.0, doppler_rate=0.0):
        self.R.rr_set_freq(ch, freq, doppler, doppler_rate)

    def write(self, x) -> int:
        if self.in_type == KO_REAL:
            return self.R.rr_write_real(np.ascontiguousarray(x, np.float32), len(x))
        return self.R.rr_write_complex(np.ascontiguousarray(x, np.complex64), len(x))

    def spectrum(self) -> np.ndarray:
        out = np.empty(self.R.rr_master_bins(), np.complex64)
        self.R.rr_get_spectrum(out)
        return out

    def downconvert(self, ch):
        """-> dict(baseband, bb_power, n0, shift, remainder)"""
        y = np.empty(self.olen[ch], np.complex64)
        p, n0, rem, sh = C.c_double(0), C.c_double(0), C.c_double(0), C.c_int(0)
        r = self.R.rr_downconvert(ch, y, C.byref(p), C.byref(n0), C.byref(sh), C.byref(rem))
        if r != 0:
            raise RuntimeError("downconvert returned %d" % r)
        return dict(baseband=y, bb_power=p.value, n0=n0.value, shift=sh.value, remainder=rem.value)

    def close(self):
        self.R.rr_close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
