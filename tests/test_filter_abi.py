"""The reference-facing surface: libka9qgpu.so behind ka9q-radio's filter.h.

CPU part: struct layouts of include/ka9q_gpu_filter.h equal the reference's own src/filter.h
(offset report produced by the same C driver compiled against either header; the reference's is
stored in tests/golden/filter_h_layout.txt).
GPU part: the driver exercises create_filter_input/output, write_*filter, set_filter,
execute_filter_output exactly as radiod does and is compared with the oracle; the variant of
the driver compiled against the REFERENCE header (oracle/_ref/driver_refhdr.so, built by
oracle/Makefile where the reference's sources are) proves the untouched sources bind unchanged.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
DRIVERS = {"driver_gpuhdr.so": ROOT / "tests" / "abi" / "_build", "driver_refhdr.so": ROOT / "oracle" / "_ref"}
TOL = 1e-5


def _build():
    subprocess.run(["make", "-C", str(ROOT / "tests" / "abi"), "-s"], check=True)


def _load(name):
    _build()
    p = DRIVERS[name] / name
    if not p.exists():
        return None
    from oracle import oracle as O

    lib = O.bind_driver(C.CDLL(str(p)))
    lib.ref_layout_report.argtypes = [C.c_char_p, C.c_int]
    lib.ref_write_real_inplace.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"), C.c_int]
    lib.ref_channel_sample_index.argtypes = [C.c_void_p, C.c_int]
    lib.ref_channel_sample_index.restype = C.c_ulonglong
    lib.ref_threaded_run.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"), C.c_int,
                                     C.c_void_p, C.c_void_p]
    f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    c64p = np.ctypeslib.ndpointer(np.complex64, flags="C_CONTIGUOUS")
    lib.ref_set_beam.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_double] * 4
    lib.ref_execute_channel_real.argtypes = [C.c_void_p, C.c_int, C.c_int, f32p]
    lib.ref_lap_probe.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, c64p]
    lib.ref_lap_probe.restype = C.c_uint
    lib.ref_produce_from_thread.argtypes = [C.c_void_p, f32p, C.c_int]
    lib.ref_channel_next_job.argtypes = [C.c_void_p, C.c_int]
    lib.ref_channel_next_job.restype = C.c_uint
    if hasattr(lib, "ref_execute_tuned"):
        lib.ref_execute_tuned.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, c64p, C.POINTER(C.c_double)]
        lib.ref_enable_noise.argtypes = [C.c_void_p, C.c_double]
        lib.ref_noise.argtypes = [C.c_void_p, C.c_int]
        lib.ref_noise.restype = C.c_double
        lib.ref_execute_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.ref_write_i16_inplace.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS"), C.c_int, C.c_float]
    if hasattr(lib, "ref_write_i16"):
        lib.ref_write_i16.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.int16, flags="C_CONTIGUOUS"), C.c_int, C.c_float, C.c_int]
    return lib


def _report(lib):
    buf = C.create_string_buffer(8192)
    lib.ref_layout_report(buf, 8192)
    return buf.value.decode()


def test_struct_layout_matches_reference_header():
    ours = _load("driver_gpuhdr.so")
    ref = (ROOT / "tests" / "golden" / "filter_h_layout.txt").read_text()   # x86-64 Linux, glibc
    assert _report(ours) == ref
    assert "filter_in.fdomain" in _report(ours)


# ------------------------------------------------------------------ GPU behaviour ---------------
@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["driver_gpuhdr.so", "driver_refhdr.so"])
def test_radiod_style_flow_matches_oracle(oracle, cuda_dev, driver, monkeypatch):
    monkeypatch.setenv("KA9Q_GPU_SPECTRUM_D2H", "all")   # this test reads the WHOLE of master->fdomain[]
    lib = _load(driver)
    if lib is None:
        pytest.skip(f"{driver} not built")
    L, M = 48000, 12001
    x = oracle.siggen_real(5 * L, 10 ** (-20 / 20), 10 ** (-40 / 20), 0.25, 10 ** (3 / 20))
    chans = [dict(olen=480, shift=15000, low=-1 / 3, high=1 / 3, beta=11.0),
             dict(olen=480, shift=-15000, low=-1 / 3, high=1 / 3, beta=11.0),
             dict(olen=240, shift=14990, low=0.01, high=0.25, beta=11.0),
             dict(olen=960, shift=15010, low=-0.2, high=0.2, beta=7.0, isb=True)]
    got, gspec = oracle.ref_run_stream(x, L, M, chans, notch_bins=[77], keep_spectra=True, lib=lib)
    ref, rspec = oracle.run_stream(x, L, M, chans, notch_bins=[77], keep_spectra=True)
    for b in range(5):
        assert np.abs(gspec[b] - rspec[b]).max() / np.abs(rspec[b]).max() < TOL   # master->fdomain[] on the host
        for c in range(len(chans)):
            assert np.abs(got[b][c] - ref[b][c]).max() / np.abs(ref[b][c]).max() < TOL, (b, c)


@pytest.mark.gpu
def test_default_spectrum_readback_covers_what_estimate_noise_reads(oracle, cuda_dev, monkeypatch):
    """Default KA9Q_GPU_SPECTRUM_D2H=windows: master->fdomain[] holds, for every slave, the >= 1000 bins around |shift| that
    the untouched estimate_noise() (radio.c:1805-1836) reads -- checked by running the oracle's restatement of it on the
    host copy -- without copying the other 1.6 M bins."""
    monkeypatch.delenv("KA9Q_GPU_SPECTRUM_D2H", raising=False)
    lib = _load("driver_gpuhdr.so")
    L, M, fs = 48000, 12001, 2.4e6
    x = oracle.siggen_real(4 * L, 0.1, 0.02, 0.25, 1.0)
    shifts = [15000, -9000, 300, 29900]
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        ids = [s.add_channel(480, -1 / 3, 1 / 3, 11.0) for _ in shifts]
        for b in range(4):
            assert s.write(x[b * L:(b + 1) * L]) == 1
            for i, sh in zip(ids, shifts):
                s.execute(i, sh)
            host = s.spectrum()
            X = oracle.forward(oracle.block_window(x, L, M, b))
            if b >= 1:   # the windows follow the shifts the slaves used on the previous block
                for sh in shifts:
                    a = oracle.estimate_noise(oracle.KO_REAL, host, 600, sh, fs)
                    r = oracle.estimate_noise(oracle.KO_REAL, X, 600, sh, fs)
                    assert abs(a - r) / r < 1e-5
                assert not host[20000:25000].any()   # far from every channel: never copied


@pytest.mark.gpu
def test_retune_filter_change_and_bookkeeping(oracle, cuda_dev):
    """Shift and filter changes between blocks take the recompute path and then rejoin the batch;
    sample_index, block_drops and the no-response / lap semantics follow filter.c."""
    lib = _load("driver_gpuhdr.so")
    L, M = 4800, 1201
    N = L + M - 1
    nb = 8
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.31, 1.0)
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        a = s.add_channel(48, -0.3, 0.3, 9.0)
        b = s.add_channel(96, -0.2, 0.4, 5.0)
        shifts_a = [1800, 1800, 1801, 1801, -1801, -1801, 1800, 1800]
        for blk in range(nb):
            if blk == 4:
                lib.ref_retune_channel(s.h, b, -0.1, 0.1, 11.0)
            assert lib.ref_write_real_inplace(s.h, x[blk * L:(blk + 1) * L], L) == 1
            ya = s.execute(a, shifts_a[blk])
            yb = s.execute(b, 1700)
            assert lib.ref_channel_sample_index(s.h, a) == blk * L
            X = oracle.forward(oracle.block_window(x, L, M, blk))
            Ra = oracle.design_response(60, 48, N, True, -0.3, 0.3, 9.0)
            Rb = oracle.design_response(120, 96, N, True, *((-0.2, 0.4, 5.0) if blk < 4 else (-0.1, 0.1, 11.0)))
            ra = oracle.channel_block(oracle.KO_REAL, X, Ra, shifts_a[blk])[-48:]
            rb = oracle.channel_block(oracle.KO_REAL, X, Rb, 1700)[-96:]
            assert np.abs(ya - ra).max() / np.abs(ra).max() < TOL, blk
            assert np.abs(yb - rb).max() / np.abs(rb).max() < TOL, blk
        assert lib.ref_channel_drops(s.h, a) == 0


@pytest.mark.gpu
def test_channel_threads_like_radiod(oracle, cuda_dev):
    """One pthread per channel blocking in execute_filter_output while a producer writes through
    the ring pointer (radio.c:996,1460; rx888.c:800-826): no drops, outputs equal the oracle."""
    lib = _load("driver_gpuhdr.so")
    L, M, nb, nch = 48000, 12001, 6, 48
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.2, 1.0)
    chans = [dict(olen=480, shift=9000 + 400 * i, low=-1 / 3, high=1 / 3, beta=11.0) for i in range(nch)]
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        for ch in chans:
            s.add_channel(ch["olen"], ch["low"], ch["high"], ch["beta"])
        outs = [np.zeros(nb * 480, np.complex64) for _ in range(nch)]
        ptrs = (C.c_void_p * nch)(*[o.ctypes.data for o in outs])
        shifts = (C.c_int * nch)(*[ch["shift"] for ch in chans])
        drops = lib.ref_threaded_run(s.h, x, nb, C.cast(shifts, C.c_void_p), C.cast(ptrs, C.c_void_p))
    assert drops == 0
    ref, _ = oracle.run_stream(x, L, M, chans)
    for c in range(nch):
        for b in range(nb):
            r = ref[b][c]
            assert np.abs(outs[c][b * 480:(b + 1) * 480] - r).max() / np.abs(r).max() < TOL, (c, b)


@pytest.mark.gpu
def test_write_i16filter_extension(oracle, cuda_dev):
    lib = _load("driver_gpuhdr.so")
    L, M, nb = 48000, 12001, 3
    f = [0.25, 0.1]
    xi = oracle.siggen_tones_i16(nb * L, f, [0.1, 0.05], 0.01, 1)
    scale = np.float32(10 ** (3 / 20) / 32768)
    xf, _, _ = oracle.convert_i16(xi, scale)
    ch = dict(olen=480, shift=15000, low=-1 / 3, high=1 / 3, beta=11.0)
    ref, _ = oracle.run_stream(xf, L, M, [ch])
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        c = s.add_channel(480, -1 / 3, 1 / 3, 11.0)
        for b in range(nb):
            # ragged writes, as USB transfers would deliver them
            blk = xi[b * L:(b + 1) * L]
            fired = 0
            for lo, hi in ((0, 16384), (16384, 40000), (40000, L)):
                fired += lib.ref_write_i16(s.h, np.ascontiguousarray(blk[lo:hi]), hi - lo, float(scale), 0)
            assert fired == 1
            y = s.execute(c, 15000)
            assert np.abs(y - ref[b][0]).max() / np.abs(ref[b][0]).max() < TOL


@pytest.mark.gpu
def test_error_conventions(oracle, cuda_dev):
    lib = _load("driver_gpuhdr.so")
    assert not lib.ref_open(0, 5, oracle.KO_REAL, 0)            # L <= 0
    assert not lib.ref_open(4801, 1201, oracle.KO_REAL, 0)      # odd L for a REAL master: unsupported, -1
    s = oracle.RefSession(4800, 1201, oracle.KO_REAL, lib=lib)
    with pytest.raises(RuntimeError):
        s.add_channel(47, -0.3, 0.3, 5.0)                        # 47*6000 % 4800 != 0 (filter.c:312-316)
    s.close()
    s = oracle.RefSession(4000, 1001, oracle.KO_REAL, lib=lib)     # N = 5000: 60*5000/4000 = 75 points
    with pytest.raises(RuntimeError):
        s.add_channel(60, 0.1, 0.3, 5.0, out_type=oracle.KO_REAL)    # odd point count: no c2r plan here (documented)
    s.close()


@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["driver_gpuhdr.so", "driver_refhdr.so"])
def test_lapped_slave_gets_zeros_and_a_drop(oracle, cuda_dev, driver):
    """filter.c:690-701: a consumer that fell >= ND blocks behind receives a block of zeros, block_drops++ and moves on
    one job -- then catches up block by block (each further call is still lapped until it is within ND)."""
    lib = _load(driver)
    if lib is None:
        pytest.skip(f"{driver} not built")
    L, M = 4800, 1201
    N = L + M - 1
    nb = 9
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.31, 1.0)
    R = oracle.design_response(60, 48, N, True, -0.3, 0.3, 9.0)
    with oracle.RefSession(L, M, oracle.KO_REAL, nworkers=1, lib=lib) as s:   # not inline: producer != consumer thread
        a = s.add_channel(48, -0.3, 0.3, 9.0)
        assert lib.ref_produce_from_thread(s.h, x[: 2 * L], 2) == 0
        y = np.empty(48, np.complex64)
        for blk in range(2):                                                   # in step: blocks 0 and 1
            assert lib.ref_lap_probe(s.h, a, 1800, None, 0, y) == 0
            X = oracle.forward(oracle.block_window(x, L, M, blk))
            r = oracle.channel_block(oracle.KO_REAL, X, R, 1800)[-48:]
            assert np.abs(y - r).max() / np.abs(r).max() < TOL
        assert lib.ref_produce_from_thread(s.h, np.ascontiguousarray(x[2 * L: 8 * L]), 6) == 0   # jobs 2..7 issued, consumer at 2
        # slot 2 now holds job 6: 4 = ND blocks ahead -> lapped
        y[:] = 1
        assert lib.ref_lap_probe(s.h, a, 1800, None, 0, y) == 1
        assert not y.any() and lib.ref_channel_next_job(s.h, a) == 3
        y[:] = 1
        assert lib.ref_lap_probe(s.h, a, 1800, None, 0, y) == 2             # job 3: slot 3 holds job 7 -> lapped again
        assert not y.any()
        for blk in (4, 5, 6, 7):                                               # back inside the ring: real data again
            assert lib.ref_lap_probe(s.h, a, 1800, None, 0, y) == 2
            X = oracle.forward(oracle.block_window(x, L, M, blk))
            r = oracle.channel_block(oracle.KO_REAL, X, R, 1800)[-48:]
            assert np.abs(y - r).max() / np.abs(r).max() < TOL, blk


@pytest.mark.gpu
@pytest.mark.parametrize("driver", ["driver_gpuhdr.so", "driver_refhdr.so"])
def test_real_output_and_beam_slaves_through_filter_h(oracle, cuda_dev, driver):
    """wfm.c:76-77 / stereod.c:387-389 create REAL slaves on a REAL master; filter.c:756-775 beam slaves on a COMPLEX one."""
    lib = _load(driver)
    if lib is None:
        pytest.skip(f"{driver} not built")
    L, M, nb = 4800, 1201, 3
    N = L + M - 1
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.0123, 1.0)
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        mono = s.add_channel(480, 50 / 24000, 0.3125, 11.0, out_type=oracle.KO_REAL)
        pilot = s.add_channel(480, -100 / 24000, 100 / 24000, 11.0)
        Rm = oracle.design_response_realout(600, 480, N, True, 50 / 24000, 0.3125, 11.0)
        Rp = oracle.design_response(600, 480, N, True, -100 / 24000, 100 / 24000, 11.0)
        for b in range(nb):
            assert s.write(x[b * L:(b + 1) * L]) == 1
            X = oracle.forward(oracle.block_window(x, L, M, b))
            y = np.empty(480, np.float32)
            assert lib.ref_execute_channel_real(s.h, mono, 0, y) == 0
            r = oracle.channel_block_realout(oracle.KO_REAL, X, Rm, 0)[-480:]
            assert np.abs(y - r).max() / np.abs(r).max() < TOL
            yp = s.execute(pilot, 59)
            rp = oracle.channel_block(oracle.KO_REAL, X, Rp, 59)[-480:]
            assert np.abs(yp - rp).max() / np.abs(rp).max() < TOL
    L, M = 4000, 1001
    N = L + M - 1
    xc = oracle.siggen_complex(nb * L, 0.1, 0.02, 0.0123, 1.0)
    with oracle.RefSession(L, M, oracle.KO_COMPLEX, lib=lib) as s:
        a = s.add_channel(480, -0.3, 0.35, 11.0)
        lib.ref_set_beam(s.h, a, 1, 0.6, -0.2, 0.3, 0.7)
        R = oracle.design_response(600, 480, N, False, -0.3, 0.35, 11.0)
        for b in range(nb):
            assert s.write(xc[b * L:(b + 1) * L]) == 1
            X = oracle.forward(oracle.block_window(xc, L, M, b))
            y = s.execute(a, 615)
            r = oracle.channel_block_beam(X, R, 615, 0.6 - 0.2j, 0.3 + 0.7j)[-480:]
            assert np.abs(y - r).max() / np.abs(r).max() < TOL


@pytest.mark.gpu
def test_tuned_output_noise_and_batch_extensions(oracle, cuda_dev):
    """execute_filter_output_tuned (radio.c:1476-1520 on the device), filter_noise_estimate (radio.c:1783-1866),
    execute_filter_output_batch and multi-block writes (k blocks per launch), against the oracle."""
    lib = _load("driver_gpuhdr.so")
    L, M, fs = 48000, 12001, 2.4e6
    N = L + M - 1
    nb = 10
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.1234, 1.0)
    freqs = [[300_017.3, 412_234.5] for _ in range(nb)]
    for b in range(5, nb):
        freqs[b][0] = 303_350.6
    R = [oracle.design_response(600, 480, N, True, -1 / 3, 1 / 3, 11.0), oracle.design_response(300, 240, N, True, 0.01, 0.25, 11.0)]
    rate = [24000.0, 12000.0]
    olen = [480, 240]
    fts = [oracle.FineTune(L, M, r) for r in rate]
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s:
        ids = [s.add_channel(480, -1 / 3, 1 / 3, 11.0), s.add_channel(240, 0.01, 0.25, 11.0)]
        assert lib.ref_enable_noise(s.h, fs) == 0
        for b in range(nb):
            assert s.write(x[b * L:(b + 1) * L]) == 1
            X = oracle.forward(oracle.block_window(x, L, M, b))
            for i in range(2):
                rc, shift, rem = oracle.compute_tuning(N, fs, freqs[b][i])
                y = np.empty(olen[i], np.complex64)
                pw = C.c_double(0)
                assert lib.ref_execute_tuned(s.h, ids[i], shift, rem, rate[i], 0.0, y, C.byref(pw)) == 0
                r = oracle.channel_block(oracle.KO_REAL, X, R[i], shift)[-olen[i]:].copy()
                p_ref = fts[i].block(r, shift, rem)
                assert np.abs(y - r).max() / np.abs(r).max() < TOL, (b, i)
                assert abs(pw.value - p_ref) / p_ref < TOL, (b, i)
                n0 = lib.ref_noise(s.h, ids[i])
                if not np.isnan(n0):   # NAN only for the blocks recomputed alone right after a (re)tune
                    ref_n0 = oracle.estimate_noise(oracle.KO_REAL, X, len(R[i]), shift, fs)
                    assert abs(n0 - ref_n0) / ref_n0 < 1e-5, (b, i)
                else:
                    assert b in (0, 5)
    # multi-block writes + batch delivery (a separate consumer thread is not needed: inline mode takes the latest job,
    # so drive it with a worker-mode session and a producer thread)
    chans = [dict(olen=480, shift=9000 + 400 * i, low=-1 / 3, high=1 / 3, beta=11.0) for i in range(24)]
    ref, _ = oracle.run_stream(x[: 6 * L], L, M, chans)
    with oracle.RefSession(L, M, oracle.KO_REAL, nworkers=1, lib=lib) as s:
        for ch in chans:
            s.add_channel(ch["olen"], ch["low"], ch["high"], ch["beta"])
        shifts = (C.c_int * 24)(*[ch["shift"] for ch in chans])
        outs = [np.zeros(480, np.complex64) for _ in range(24)]
        ptrs = (C.c_void_p * 24)(*[o.ctypes.data for o in outs])
        # first pass establishes the shifts (recompute path), then 3 blocks arrive in ONE write: one launch of 3 blocks
        assert lib.ref_produce_from_thread(s.h, np.ascontiguousarray(x[:L]), 1) == 0
        assert lib.ref_execute_batch(s.h, C.cast(shifts, C.c_void_p), C.cast(ptrs, C.c_void_p)) == 0
        for c in range(24):
            assert np.abs(outs[c] - ref[0][c]).max() / np.abs(ref[0][c]).max() < TOL
        big = np.ascontiguousarray(x[L: 4 * L])
        lib.ref_write_real.argtypes = [C.c_void_p, np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS"), C.c_int]

        class _W(C.Structure):
            pass
        import threading

        t = threading.Thread(target=lambda: lib.ref_write_real(s.h, big, 3 * L))
        t.start()
        t.join()
        for b in (1, 2, 3):
            assert lib.ref_execute_batch(s.h, C.cast(shifts, C.c_void_p), C.cast(ptrs, C.c_void_p)) == 0
            for c in range(24):
                assert np.abs(outs[c] - ref[b][c]).max() / np.abs(ref[b][c]).max() < TOL, (b, c)
        assert sum(lib.ref_channel_drops(s.h, c) for c in range(24)) == 0


@pytest.mark.gpu
def test_secondary_complex_master_like_filter2(oracle, cuda_dev):
    """radio.c:1572-1602 / :1503-1514: a channel's output is written into a second, small COMPLEX master (`filter2`) with
    write_cfilter, run inline by the same thread (perform_inline, owner shortcut filter.c:681-683), and read back with shift 0.
    Both masters live in the same library at the same time."""
    lib = _load("driver_gpuhdr.so")
    L, M, nb = 48000, 12001, 6
    x = oracle.siggen_real(nb * L, 0.1, 0.02, 0.25, 1.0)
    ch = dict(olen=480, shift=15000, low=-1 / 3, high=1 / 3, beta=11.0)
    first, _ = oracle.run_stream(x, L, M, [ch])
    mid = np.concatenate([first[b][0] for b in range(nb)]).astype(np.complex64)
    L2, M2 = 480, 97   # blocking = 1: N = 576 = 2^6 * 9
    ch2 = dict(olen=480, shift=0, low=-0.125, high=0.125, beta=7.0)
    second, _ = oracle.run_stream(mid, L2, M2, [ch2])
    with oracle.RefSession(L, M, oracle.KO_REAL, lib=lib) as s1, oracle.RefSession(L2, M2, oracle.KO_COMPLEX, lib=lib) as s2:
        a = s1.add_channel(480, -1 / 3, 1 / 3, 11.0)
        b2 = s2.add_channel(480, -0.125, 0.125, 7.0)
        for b in range(nb):
            assert s1.write(x[b * L:(b + 1) * L]) == 1
            y = s1.execute(a, 15000)
            assert np.abs(y - first[b][0]).max() / np.abs(first[b][0]).max() < TOL
            assert s2.write(y) == 1
            z = s2.execute(b2, 0)
            r = second[b][0]
            assert np.abs(z - r).max() / np.abs(r).max() < 2 * TOL, b   # two cascaded float32 filters
