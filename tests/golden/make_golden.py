#!/usr/bin/env python3
"""Generate tests/golden/*.npz by running the REFERENCE's own filter.c (oracle/_ref, compiled
unmodified from /root/reference/src by oracle/Makefile) -- the reference ships no golden vectors
or tests of its own (SURVEY.md section 4), so these fixtures are its outputs captured here.

Needs oracle/_ref (make -C oracle REFERENCE=<ka9q-radio checkout>):
    python tests/golden/make_golden.py [fixture ...]        (default: every fixture)
The fixtures are small on purpose; the input streams are regenerated from the stored sig_gen
parameters (the restated generator is bit-exact with sig_gen.c/gauss.c/osc.c, which the fixture
also pins via a few raw samples and a float64 checksum).  Long vectors are stored as every k-th
entry (the `*stride` keys) plus their last TAIL entries (`*_tail`), next to the largest magnitude of
the whole vector, so a test keeps the denominator of its relative error.  Each fixture also stores
the parameters it was made with; the tests that read it assert that theirs are the same.
"""
import ctypes as C
import hashlib
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import oracle as O  # noqa: E402

OUT = Path(__file__).resolve().parent
OUT_STRIDE = 3   # channel outputs, responses and baseband: every 3rd sample ...
TAIL = 4         # ... and the last 4


def _spec_stride(bins):
    return max(1, bins // 128)


CASES = {
    # name: (in_type, L, M, nblocks, siggen(amplitude, noise, cycles/sample, scale), notch bins, channels)
    "real_small": dict(
        in_type=O.KO_REAL, L=4800, M=1201, nb=4, sig=(0.1, 0.01, 0.25 + 1 / 64.0, 10 ** (3 / 20)), notch=[77],
        chans=[dict(olen=48, shift=1594, low=-1 / 3, high=1 / 3, beta=11.0),
               dict(olen=48, shift=-1594, low=-1 / 3, high=1 / 3, beta=11.0),
               dict(olen=96, shift=1590, low=0.01, high=0.3, beta=7.0),
               dict(olen=24, shift=3, low=-0.4, high=0.4, beta=3.0),
               dict(olen=48, shift=1600, low=-0.25, high=0.25, beta=11.0, isb=True)]),
    "complex_small": dict(
        in_type=O.KO_COMPLEX, L=4000, M=1001, nb=4, sig=(0.1, 0.01, -0.123, 1.0), notch=None,
        chans=[dict(olen=80, shift=-615, low=-1 / 3, high=1 / 3, beta=11.0),
               dict(olen=80, shift=2499, low=-1 / 3, high=1 / 3, beta=11.0),
               dict(olen=160, shift=-2490, low=-0.2, high=0.45, beta=5.0),
               dict(olen=40, shift=0, low=-0.5, high=0.5, beta=11.0)]),
    # cfg-1 of BASELINE.json: sig_gen real 2.4 MS/s, carrier 600 kHz at -20 dBFS, noise -40 dBFS,
    # one 24 kHz NBFM channel (preset fm: +-8 kHz, beta 11), DC notch as radio.c:601-620 installs it
    "cfg1_siggen": dict(
        in_type=O.KO_REAL, L=48000, M=12001, nb=6, sig=(10 ** (-20 / 20), 10 ** (-40 / 20), 600e3 / 2.4e6, 10 ** (3 / 20)),
        notch=[], chans=[dict(olen=480, shift=15000, low=-8000 / 24000, high=8000 / 24000, beta=11.0)]),
    # tests/test_oracle_cpu.py::test_restatement_matches_reference_library: shifts at 0, near +-N/2, both signs, ISB
    "reference_library": dict(
        in_type=O.KO_REAL, L=4800, M=1201, nb=5, sig=(0.2, 0.05, 0.3123, 1.0), notch=[5],
        chans=[dict(olen=48, shift=s, low=-0.3, high=0.4, beta=9.0) for s in (1874, -1874, 0, 2999, -3005, 2990, 12)]
        + [dict(olen=96, shift=1870, low=-0.2, high=0.2, beta=4.0, isb=True)]),
}


def make_stream(c):
    a, n, f, s = c["sig"]
    if c["in_type"] == O.KO_REAL:
        return O.ref_siggen_real(c["nb"] * c["L"], a, n, f, s)
    return O.ref_siggen_complex(c["nb"] * c["L"], a, n, f, s)


def stream_case(name):
    c = CASES[name]
    x = make_stream(c)
    outs, specs = O.ref_run_stream(x, c["L"], c["M"], c["chans"], notch_bins=c["notch"], keep_spectra=True)
    with O.RefSession(c["L"], c["M"], c["in_type"]) as s:
        resp = [s.response(s.add_channel(ch["olen"], ch["low"], ch["high"], ch["beta"])) for ch in c["chans"]]
    data = dict(
        in_type=c["in_type"], L=c["L"], M=c["M"], nb=c["nb"], sig=np.array(c["sig"], np.float64),
        notch=np.array(c["notch"] if c["notch"] is not None else [-1], np.int64),
        chan_params=np.array([[ch["olen"], ch["shift"], ch["low"], ch["high"], ch["beta"], float(ch.get("isb", False))]
                              for ch in c["chans"]], np.float64),
        x_head=x[:16].copy(), x_sum=np.array([np.sum(x.astype(np.complex128))]),
        x_sha=np.frombuffer(hashlib.sha256(x.tobytes()).digest(), np.uint8),
    )
    stride = max(1, len(specs[0]) // 512)
    data["spec_stride"] = stride
    data["spec_sub"] = np.stack([sp[::stride] for sp in specs])
    data["spec_absmax"] = np.array([np.abs(sp).max() for sp in specs])
    data["spec_sum"] = np.array([np.sum(sp.astype(np.complex128)) for sp in specs])
    data["spec_energy"] = np.array([np.sum(np.abs(sp.astype(np.complex128)) ** 2) for sp in specs])
    for i in range(len(c["chans"])):
        data[f"out{i}"] = np.stack([outs[b][i] for b in range(c["nb"])])
        data[f"resp{i}"] = resp[i]
    _save(name, data)


def _sub(v, stride):
    """(every stride-th entry, the last TAIL entries) of one vector"""
    return v[::stride], v[-TAIL:]


def _stack(data, key, pairs):
    """pairs of _sub() per block -> data[key] and data[key + "_tail"]"""
    data[key] = np.stack([p[0] for p in pairs])
    data[key + "_tail"] = np.stack([p[1] for p in pairs])


def _save(name, data):
    np.savez_compressed(OUT / f"{name}.npz", **data)
    print(name, "written", sum(v.nbytes for v in data.values() if hasattr(v, "nbytes")) // 1024, "KiB raw")


def _source_bins(X, R, fd):
    """The master bin every entry of one reference slice was taken from: fd[j] == X[k] R[j] -> k + 1,
    conj(X[k]) R[j] -> -(k + 1), 0 -> 0.  Checked against fd before it is stored."""
    X, R = X.astype(np.complex128), R.astype(np.complex128)
    plain = np.abs(fd[:, None] - R[:, None] * X[None, :])
    conj = np.abs(fd[:, None] - R[:, None] * np.conj(X)[None, :])
    kp, kc = plain.argmin(1), conj.argmin(1)
    j = np.arange(len(fd))
    src = np.where(plain[j, kp] <= conj[j, kc], kp + 1, -(kc + 1))
    src[fd == 0] = 0
    assert np.abs(O.rebuild_slice(X, R, src) - fd).max() <= 1e-7 * np.abs(fd).max() + 1e-12
    return src.astype(np.int16)


SWEEP_OLENS = (48, 24, 40)


def slice_sweep():
    """tests/test_oracle_cpu.py::test_slice_sweep_matches_reference_library: every integer shift, REAL and COMPLEX masters,
    even and odd slave sizes.  The reference's master spectrum and responses are stored, each slice as its source bins."""
    data = {"olens": np.array(SWEEP_OLENS)}
    for tag, in_type, L, M in (("real", O.KO_REAL, 480, 121), ("complex", O.KO_COMPLEX, 480, 121)):
        N = L + M - 1
        rng = np.random.default_rng(7)
        x = (rng.standard_normal(L) + (1j * rng.standard_normal(L) if in_type == O.KO_COMPLEX else 0))
        x = x.astype(np.complex64 if in_type == O.KO_COMPLEX else np.float32)
        with O.RefSession(L, M, in_type) as s:
            ids = [s.add_channel(olen, -0.3, 0.3, 8.0) for olen in SWEEP_OLENS]
            s.write(x)
            X = s.spectrum()
            data[f"{tag}_X"] = X
            lim = N // 2 if in_type == O.KO_COMPLEX else N
            for i in ids:
                R = s.response(i)
                data[f"{tag}_R{i}"] = R
                data[f"{tag}_src{i}"] = np.stack([_source_bins(X, R, s.execute(i, shift, want_fdomain=True)[1])
                                                  for shift in range(-lim + 1, lim)])
    _save("slice_sweep", data)


OSC_CASES = [(0.0123, 0.0), (-0.25, 0.0), (1e-3, 1e-9), (0.0, 0.0)]
OSC_N = 40000


def osc_samples():
    """tests/test_oracle_ext_cpu.py::test_osc_restatement_vs_reference_osc: osc.c's recursive oscillator over 40000 steps
    (two renormalisations, every 16384 steps), stored every 199th step and around each renormalisation."""
    idx = np.array(sorted(set(range(0, OSC_N, 199)) | set(range(16380, 16390)) | set(range(32764, 32774))
                          | set(range(OSC_N - 4, OSC_N))), np.int64)
    data = {"idx": idx, "cases": np.array(OSC_CASES)}
    for k, (f, r) in enumerate(OSC_CASES):
        ref = np.empty(OSC_N, np.complex128)
        O.radio_lib().rr_osc_run(f, r, OSC_N, ref.ctypes.data)
        data[f"osc{k}"] = ref[idx]
    _save("osc_samples", data)


DOWNCONVERT = {
    # name: (in_type, L, M, fs, front-end frequency, chans (olen, out rate, low, high, beta), blocks, carrier per block and channel)
    "downconvert_real": (O.KO_REAL, 4800, 1201, 240e3, 0.0,
                         [(480, 24000.0, -1 / 3, 1 / 3, 11.0), (240, 12000.0, 50 / 12000, 3000 / 12000, 11.0),
                          (960, 48000.0, -0.4, 0.4, 7.0)], 9,
                         [[33_333.3 if b >= 4 else 30_017.3, 61_234.5 + 7.25 if b >= 6 else 61_234.5, 90_000.0] for b in range(9)]),
    "downconvert_complex": (O.KO_COMPLEX, 4000, 1001, 200e3, 10.0e6,
                            [(480, 24000.0, -1 / 3, 1 / 3, 11.0), (480, 24000.0, -0.3, 0.2, 9.0)], 7,
                            [[10.0e6 + 23_456.7, 10.0e6 - 12_000.0 if b >= 3 else 10.0e6 - 41_234.5] for b in range(7)]),
}


def downconvert(name):
    """tests/test_oracle_ext_cpu.py::test_downconvert_*_vs_reference_radio: radio.c's downconvert() per block and channel."""
    in_type, L, M, fs, fe_freq, chans, nb, plan = DOWNCONVERT[name]
    if in_type == O.KO_REAL:
        x = O.siggen_real(nb * L, 0.1, 0.02, 0.1234, 1.0)
    else:
        x = O.siggen_complex(nb * L, 0.1, 0.02, 0.1234, 1.0)
    keys = ("shift", "remainder", "bb_power", "n0")
    rows = {k: [] for k in keys + ("bb_absmax", "spec_absmax")}
    spec_sub = []
    bb = [[] for _ in chans]
    with O.RadioRef(L, M, in_type, fs, fe_freq) as rr:
        ids = [rr.add_channel(c[0], c[1], plan[0][i], c[2], c[3], c[4]) for i, c in enumerate(chans)]
        for b in range(nb):
            assert rr.write(x[b * L:(b + 1) * L]) == 1
            spec = rr.spectrum()
            spec_sub.append(_sub(spec, _spec_stride(len(spec))))
            rows["spec_absmax"].append(np.abs(spec).max())
            d = []
            for i in range(len(chans)):
                rr.set_freq(ids[i], plan[b][i])
                d.append(rr.downconvert(ids[i]))
                bb[i].append(_sub(d[i]["baseband"], OUT_STRIDE))
            for k in keys:
                rows[k].append([di[k] for di in d])
            rows["bb_absmax"].append([np.abs(di["baseband"]).max() for di in d])
    data = {k: np.array(v) for k, v in rows.items()}
    _stack(data, "spec_sub", spec_sub)
    for i, v in enumerate(bb):
        _stack(data, f"bb{i}", v)
    data.update(plan=np.array(plan), chans=np.array(chans), spec_stride=_spec_stride(len(spec)), stride=OUT_STRIDE)
    _save(name, data)


REALOUT_CASES = [(480, 50 / 24000, 0.3, 11.0, 0), (960, 0.01, 0.45, 7.0, 0), (480, -0.2, 0.25, 11.0, 40), (240, 0.05, 0.3, 5.0, -7)]
BEAM_CASES = [(480, 615, 1.0, 0.0), (480, -615, 0.0, 1.0), (160, 300, 0.6 - 0.2j, 0.3 + 0.7j), (80, 0, 1.0, 1j),
              (480, 2100, 0.5, -0.5j), (480, -2150, 0.2j, 0.9)]


def _ref_exec(s, ch, shift, olen, real_out):
    n = s.R.ref_channel_points(s.h, ch)
    dt = np.float32 if real_out else np.complex64
    dst, full = np.empty(olen, dt), np.empty(n, dt)
    assert s.R.ref_execute_channel(s.h, ch, int(shift), dst.ctypes.data, full.ctypes.data, None) == 0
    return dst, full


def realout():
    """tests/test_oracle_ext_cpu.py::test_realout_slaves_vs_reference_library: REAL-output slaves on both master types."""
    data = {"stride": OUT_STRIDE, "cases": np.array(REALOUT_CASES)}
    L, M, nb = 4800, 1201, 3
    for tag, it in (("real", O.KO_REAL), ("complex", O.KO_COMPLEX)):
        if it == O.KO_REAL:
            x = O.siggen_real(nb * L, 0.1, 0.02, 0.0123, 1.0)
        else:
            x = O.siggen_complex(nb * L, 0.1, 0.02, 0.0123, 1.0)
        full_sub = [[] for _ in REALOUT_CASES]
        full_max = []
        with O.RefSession(L, M, it) as s:
            ids = [s.add_channel(c[0], c[1], c[2], c[3], out_type=O.KO_REAL) for c in REALOUT_CASES]
            for i in ids:
                r = s.response(i)
                r = r[: len(r) // 2 + 1]
                data[f"{tag}_resp{i}"], data[f"{tag}_resp{i}_tail"] = _sub(r, OUT_STRIDE)
                data[f"{tag}_resp_absmax{i}"] = np.abs(r).max()
            for b in range(nb):
                assert s.write(x[b * L:(b + 1) * L]) == 1
                row = []
                for i, c in zip(ids, REALOUT_CASES):
                    dst, full = _ref_exec(s, i, c[4], c[0], True)
                    assert np.array_equal(full[-c[0]:], dst)   # the user-visible part is the last olen samples
                    full_sub[i].append(_sub(full, OUT_STRIDE))
                    row.append(np.abs(full).max())
                full_max.append(row)
        for i, v in enumerate(full_sub):
            _stack(data, f"{tag}_full{i}", v)
        data[f"{tag}_full_absmax"] = np.array(full_max)
    _save("realout", data)


def beam():
    """tests/test_oracle_ext_cpu.py::test_beam_slaves_vs_reference_library: beam slaves on a COMPLEX master."""
    L, M, nb = 4000, 1001, 3
    x = O.siggen_complex(nb * L, 0.1, 0.02, 0.0123, 1.0)
    dst_sub = [[] for _ in BEAM_CASES]
    dst_max = []
    with O.RefSession(L, M, O.KO_COMPLEX) as s:
        s.R.ref_set_beam.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 4
        ids = [s.add_channel(c[0], -0.3, 0.35, 11.0) for c in BEAM_CASES]
        for i, c in zip(ids, BEAM_CASES):
            s.R.ref_set_beam(s.h, i, 1, complex(c[2]).real, complex(c[2]).imag, complex(c[3]).real, complex(c[3]).imag)
        for b in range(nb):
            assert s.write(x[b * L:(b + 1) * L]) == 1
            row = []
            for i, c in zip(ids, BEAM_CASES):
                dst, _ = _ref_exec(s, i, c[1], c[0], False)
                dst_sub[i].append(_sub(dst, OUT_STRIDE))
                row.append(np.abs(dst).max())
            dst_max.append(row)
    data = {"cases": np.array(BEAM_CASES), "dst_absmax": np.array(dst_max), "stride": OUT_STRIDE}
    for i, v in enumerate(dst_sub):
        _stack(data, f"dst{i}", v)
    _save("beam", data)


def filter_h_layout():
    """tests/test_filter_abi.py::test_struct_layout_matches_reference_header: the layout report of tests/abi/filter_driver.c
    compiled against the reference's own src/filter.h (x86-64 Linux, glibc)."""
    import subprocess

    subprocess.run(["make", "-C", str(ROOT / "oracle"), "-s"], check=True)
    lib = C.CDLL(str(ROOT / "oracle" / "_ref" / "driver_refhdr.so"))
    lib.ref_layout_report.argtypes = [C.c_char_p, C.c_int]
    buf = C.create_string_buffer(8192)
    lib.ref_layout_report(buf, 8192)
    (OUT / "filter_h_layout.txt").write_text(buf.value.decode())
    print("filter_h_layout written")


FIXTURES = {**{name: (lambda n=name: stream_case(n)) for name in CASES},
            "slice_sweep": slice_sweep, "osc_samples": osc_samples,
            **{name: (lambda n=name: downconvert(n)) for name in DOWNCONVERT},
            "realout": realout, "beam": beam, "filter_h_layout": filter_h_layout}


def main(names):
    for name in names or FIXTURES:
        FIXTURES[name]()


if __name__ == "__main__":
    main(sys.argv[1:])
