#!/usr/bin/env python3
"""bench.py -- headline benchmark of the overlap-save channelizer hot path (BASELINE.json).

Metric: input Msamples/s through forward + filter + inverse at N channels.  Default workload at one GPU is cfg-2
(RX888 129.6 MS/s real int16, N = 3 240 000, 1024 x 24 kHz NBFM channels); `--config cfg3|cfg4|cfg5` select the other
BASELINE.json configurations (ka9q_radio_b200/workloads.py).  With several GPUs the default is cfg-5's channel plan
(8192 channels at f_k = 0.5 MHz + k*7.52 kHz, 1024 contiguous channels per GPU).
A "step" runs the hot path over `--blocks-per-step` consecutive 20 ms blocks.

  python bench.py --gpus 1 --steps K --warmup W          our arm (CUDA, through the C-ABI)
  python bench.py --impl reference ...                   the reference's own CPU path (oracle/_ref:
                                                         filter.c compiled unmodified + FFT shim)
  torchrun ... bench.py --gpus N                         channel groups sharded over N GPUs, forward
                                                         transform on rank 0 + one NCCL broadcast of
                                                         the spectrum per step (north_star / SURVEY 8e)
  python bench.py ... --dump-outputs DIR                 also write the channel outputs of the last timed
                                                         step to DIR (compare two builds output for output)
One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.  The GPU arm never imports the
oracle: inputs come from ka9q_radio_b200/workloads.py; the parity self-check and the CPU baseline run in subprocesses.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# the tree may be read-only: no bytecode caches next to the sources, here or in the subprocesses
sys.dont_write_bytecode = True
os.environ["PYTHONDONTWRITEBYTECODE"] = "1"

METRIC = "input Msamples/s through forward+filter+inverse at N channels"
L2_BYTES = 126e6   # B200 L2 (B200_PROFILING.md); the resident input a rank cycles through must exceed it



class ClockSampler:
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def _tone_channels(w, limit=3):
    """indices of the first few channels that carry one of the synthetic tones (the loudness reference of the parity check)"""
    hz_per_bin = w.fs / w.N
    out = []
    for i, c in enumerate(w.channels):
        if any(abs(abs(c.shift) * hz_per_bin - abs(f)) < 2000.0 and (c.shift >= 0) == (f >= 0 or w.in_type == 2) for f in w.tones_hz):
            out.append(i)
            if len(out) >= limit:
                break
    return out


def _workload(args, rank=0, world=1):
    from ka9q_radio_b200 import workloads

    name = args.config or ("cfg2" if world == 1 else "cfg5")
    return workloads.by_name(name, rank, world)


# --------------------------------------------------------------------------------------------
# the two legs that may touch oracle/: both run in a fresh subprocess
_REF_CODE = r"""
import sys, json, os, ctypes as C
sys.path.insert(0, %(root)r)
import numpy as np
from oracle import oracle as O
from ka9q_radio_b200 import workloads
w = workloads.by_name(%(cfg)r)
R = O.ref_lib()
blocks, steps, warmup, nworkers = %(blocks)d, %(steps)d, %(warmup)d, %(nworkers)d
x = w.stream(4)
if w.in_type == workloads.KGPU_REAL:
    xf, _, _ = O.convert_i16(x, np.float32(w.scale))       # what rx888.c's convert() leaves in the ring
    n_in = len(xf)
else:
    xf = (x[0::2].astype(np.float32) * np.float32(w.scale) + 1j * (x[1::2].astype(np.float32) * np.float32(w.scale))).astype(np.complex64)
    n_in = len(xf)
R.ref_bench_mixed.restype = C.c_double
R.ref_bench_mixed.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 5 + [C.c_void_p, C.c_long, C.c_int, C.c_int, C.POINTER(C.c_uint)]
n = len(w.channels)
olen = (C.c_int * n)(*[c.olen for c in w.channels])
shifts = (C.c_int * n)(*[c.shift for c in w.channels])
low = (C.c_double * n)(*[c.low for c in w.channels])
high = (C.c_double * n)(*[c.high for c in w.channels])
beta = (C.c_double * n)(*[c.beta for c in w.channels])
olens = sorted(set(c.olen for c in w.channels))
times = []
drops_total = 0
for s in range(warmup + steps):
    drops = C.c_uint(0)
    t = R.ref_bench_mixed(w.L, w.M, w.in_type, n, C.cast(olen, C.c_void_p), C.cast(shifts, C.c_void_p), C.cast(low, C.c_void_p),
                          C.cast(high, C.c_void_p), C.cast(beta, C.c_void_p), xf.ctypes.data, n_in, blocks, nworkers, C.byref(drops))
    drops_total += int(drops.value)
    if s >= warmup: times.append(t)
print(json.dumps({"times": times, "drops": drops_total, "groups": len(olens)}))
"""


def cpu_reference_run(cfg: str, blocks: int, steps: int, warmup: int) -> dict:
    """oracle/_ref (reference filter.c unmodified + fftw shim) driven as radiod drives it: one
    producer, FFT worker threads, one pthread per channel (ref_driver.c:ref_bench).  Runs in a
    fresh subprocess because filter.c starts its worker pool once per process (filter.c:1047)."""
    from ka9q_radio_b200 import workloads

    w = workloads.by_name(cfg)
    ncores = os.cpu_count() or 1
    nworkers = max(1, min(3, ncores - 1))   # ND=4 spectrum ring: at most 3 forward FFTs in flight (filter.h:48)
    code = _REF_CODE % dict(root=str(ROOT), cfg=cfg, blocks=blocks, steps=steps, warmup=warmup, nworkers=nworkers)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True)
    res = json.loads(out.stdout.strip().splitlines()[-1])
    tot = float(np.sum(res["times"]))
    value = blocks * len(res["times"]) * w.L / tot / 1e6
    fftw = "absent on this box (ldconfig lists only cuFFTW); dlopen('libfftw3f.so.3') failed"
    try:
        C.CDLL("libfftw3f.so.3")
        fftw = "present but not used by this arm"
    except OSError:
        pass
    kind = "reference" if (ROOT / "oracle" / "_ref" / "libka9qref.so").exists() else "port"
    return {"value": value, "ms_per_step": 1e3 * tot / len(res["times"]),
            "cpu_baseline": {"value": value, "unit": "Msamples/s", "cores": ncores, "kind": kind,
                             "threads": f"1 producer + {nworkers} forward-FFT workers + one thread per channel ({len(w.channels)})",
                             "fft_backend": "oracle/fft_cpu.c shim behind fftw3.h; this is NOT an FFTW-with-wisdom figure "
                                            f"(a tuned FFTW r2c is typically 2-4x faster than this shim). libfftw3f: {fftw}",
                             "sample": f"{blocks} blocks x {len(res['times'])} runs of {cfg} (float input already in the ring"
                                       + f"), {res['drops']} dropped blocks"}}


def run_reference(args) -> None:
    """The reference's own CPU implementation of the path, timed on this box's host cores."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = _workload(args, 0, 1 if args.config else max(1, args.gpus))
    cfg = w.name if w.name != "cfg5" else "cfg2"   # per-GPU share of cfg-5 == one 1024-channel bank; same CPU work as cfg-2
    res = cpu_reference_run(cfg, blocks=args.ref_blocks, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": "Msamples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.description, "blocks_per_step": args.ref_blocks},
        "cpu_baseline": res["cpu_baseline"],
        "e2e": {"value": res["value"], "unit": "Msamples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


_PARITY_CODE = r"""
import sys, json
sys.path.insert(0, %(root)r)
import numpy as np
from oracle import oracle as O
z = np.load(%(npz)r)
L, M, in_type, scale = int(z["L"]), int(z["M"]), int(z["in_type"]), np.float32(z["scale"])
N = L + M - 1
worst, checked, loud = 0.0, 0, 0.0
resp = {}
items = []
for bi in range(len(z["blocks"])):
    win = z["win%%d" %% bi]
    if in_type == O.KO_REAL:
        xf, _, _ = O.convert_i16(win, scale)
    else:
        xf = (win[0::2].astype(np.float32) * scale + 1j * (win[1::2].astype(np.float32) * scale)).astype(np.complex64)
    X = O.forward(xf)
    for ci, c in enumerate(z["chans"]):
        olen, shift, low, high, beta = int(z["olen"][ci]), int(z["shift"][ci]), float(z["low"][ci]), float(z["high"][ci]), float(z["beta"][ci])
        key = (olen, low, high, beta)
        if key not in resp:
            resp[key] = O.design_response(olen * N // L, olen, N, in_type == O.KO_REAL, low, high, beta)
        ref = O.channel_block(in_type, X, resp[key], shift)[-olen:]
        got = z["out%%d_%%d" %% (bi, ci)]
        items.append((ref, got))
        loud = max(loud, float(np.abs(ref).max()))
worst_loud = 0.0
for ref, got in items:
    # channels more than 30 dB below the loudest are measured against that level (two float32 transforms differ by
    # ~1e-7 of the strongest channel everywhere: tests/test_gpu_configs.py); loud channels against their own peak
    own = float(np.abs(ref).max())
    d = float(np.abs(got - ref).max())
    worst = max(worst, d / max(own, 3e-2 * loud))
    if own >= 0.1 * loud:
        worst = max(worst, d / own)
        worst_loud = max(worst_loud, d / own)
    checked += 1
print(json.dumps({"max_rel_err": worst, "max_rel_err_loud_channels": worst_loud, "checked": checked,
                  "measure": "max|gpu-ref| / max(max|ref|, 3e-2 * loudest channel of the check) per channel-block"}))
"""


def parity_check(w, host_stream: np.ndarray, pairs: dict, first_block: int, windows: dict | None = None) -> dict:
    """pairs: {(block in launch, channel index): complex64[olen]} pulled from the timed configuration's last step.
    Compared in a subprocess with the oracle (forward transform of the block's window + channel) at north_star's 1e-5."""
    blocks = sorted({b for b, _ in pairs})
    chans = sorted({c for _, c in pairs})
    wpb = w.samples_per_block
    hist = (w.M - 1) * (2 if w.in_type == 1 else 1)
    data = dict(L=w.L, M=w.M, in_type=w.in_type, scale=np.float32(w.scale), blocks=np.array(blocks), chans=np.array(chans),
                olen=np.array([w.channels[c].olen for c in chans]), shift=np.array([w.channels[c].shift for c in chans]),
                low=np.array([w.channels[c].low for c in chans]), high=np.array([w.channels[c].high for c in chans]),
                beta=np.array([w.channels[c].beta for c in chans]))
    padded = np.concatenate([np.zeros(hist, np.int16), host_stream])
    for bi, b in enumerate(blocks):
        g = (first_block + b) * wpb
        data[f"win{bi}"] = windows[b] if windows is not None else padded[g: g + hist + wpb].copy()
        for ci, c in enumerate(chans):
            data[f"out{bi}_{ci}"] = pairs[(b, c)]
    with tempfile.TemporaryDirectory() as td:
        npz = os.path.join(td, "parity.npz")
        np.savez(npz, **data)
        out = subprocess.run([sys.executable, "-c", _PARITY_CODE % dict(root=str(ROOT), npz=npz)], capture_output=True, text=True)
    if out.returncode != 0:
        return {"max_rel_err": None, "checked": 0, "error": out.stderr[-400:]}
    r = json.loads(out.stdout.strip().splitlines()[-1])
    r.update({"tolerance": 1e-5, "ok": r["max_rel_err"] < 1e-5, "blocks_of_launch": blocks, "first_block": first_block,
              "channels": len(chans), "against": "oracle (CPU restatement pinned to the reference's filter.c), in a subprocess"})
    return r


# --------------------------------------------------------------------------------------------
def run_ours(args) -> None:
    import torch
    import torch.distributed as dist

    from ka9q_radio_b200 import capi
    from ka9q_radio_b200.channelizer import Channelizer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the channelizer has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The forward and channel grids fill every SM; a collective's CTAs launched from a normal-priority stream only get
        # scheduled once the running grid has nothing left to dispatch, i.e. the "overlapped" collective serialises behind the
        # kernels.  NCCL's internal stream at high priority lets its few CTAs slip in as ours retire.
        opts = None
        if os.environ.get("KA9Q_NCCL_HIPRI", "1") != "0":
            try:
                opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
            except Exception:
                opts = None
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)
    lib = capi.load()
    B = args.blocks_per_step
    nstream = args.stream_blocks
    w = _workload(args, rank, world)
    L, M, N = w.L, w.M, w.N
    wpb = w.samples_per_block
    hist = (M - 1) * (2 if w.in_type == capi.KGPU_COMPLEX else 1)
    nchan = len(w.channels)

    cz = Channelizer(L, M, w.in_type, dev, capacity=nchan)
    for c in w.channels:
        cz.add_channel(c.olen, c.shift, c.low, c.high, c.beta)
    alg_bytes = cz.bank.algorithmic_bytes(capi.KGPU_FMT_I16)       # per block, SURVEY.md 8d
    alg_fwd_in = N * (4.0 if w.in_type == capi.KGPU_COMPLEX else 2.0)
    alg_fwd_out = cz.master.bins * 8.0
    alg_chan = alg_bytes - alg_fwd_in - alg_fwd_out

    # ---- inputs: a stream larger than L2, resident in HBM before the timed region ----------
    # block-parallel modes: a rank only reads B/world of a step's windows, so the resident stream is lengthened until the part
    # a rank cycles through is larger than L2 as well (8 GPUs: 256 blocks = 1.3 GB per GPU)
    rank_reads = (B // world if world > 1 and args.mg_mode in ("allgather", "a2a") else B) * wpb * 2   # bytes per step
    nstream = max(nstream, B * int(np.ceil(1.25 * L2_BYTES / rank_reads)))
    host = w.stream(nstream)
    hpin = torch.from_numpy(np.concatenate([np.zeros(hist, np.int16), host])).pin_memory()
    d_stream = hpin.to(dev)
    ngroups = nstream // B
    from ka9q_radio_b200.sharding import PipelinedSharder

    nslots = max(2, args.depth)
    spec2 = [cz.alloc_spectra(B) for _ in range(nslots)]
    out = cz.alloc_outputs(B)
    comp = torch.cuda.current_stream(dev)
    mc, mc_why = None, "single GPU"
    fwd = lambda step, slot: cz.forward(d_stream, B, spec2[slot], scale=w.scale, first_block=(step % ngroups) * B)
    chan = lambda step, slot: cz.channels(spec2[slot], B, out)
    mode = args.mg_mode if world > 1 else "single"
    if world > 1 and mode == "spectrum-mc":
        # own multicast copy kernel over NVSwitch when the fabric offers a multicast mapping
        from ka9q_radio_b200.multicast import SpectrumMulticast
        mc, mc_why = SpectrumMulticast.create(rank, world, dev, 2, B * cz.master.spec_stride * 2,
                                                  nctas=int(os.environ.get("KA9Q_MC_CTAS", "64")))
    if mc is not None:
        from ka9q_radio_b200.sharding import MulticastSharder
        symm2 = [mc.slot_view(s, (B, cz.master.spec_stride)) for s in range(2)]
        sharder = MulticastSharder(
            rank, world, forward=fwd, push=lambda slot: mc.push(slot, spec2[slot]), ready=mc.ready, arrive=mc.arrive,
            channels=lambda step, slot: cz.channels(spec2[slot] if rank == 0 else symm2[slot], B, out))
        par = (f"{world} GPUs: forward on rank 0, spectra stored once per step to an NVSwitch multicast address by "
               "kgpu_multicast_copy (own kernel, multimem.st) + symmetric-memory barrier")
    elif mode in ("spectrum", "spectrum-mc", "single"):
        # north_star: forward transform once (rank 0), ONE broadcast of the block spectra per step
        sharder = PipelinedSharder(rank, world, forward=fwd, channels=chan, depth=nslots,
                                   broadcast=lambda slot: dist.broadcast(spec2[slot], src=0, async_op=True))
        par = ("single GPU" if world == 1 else
               f"{world} GPUs: forward on rank 0, 1 NCCL broadcast of the spectrum per step ({B} blocks, {nslots}-deep ring)"
               + (f" (multicast path unavailable: {mc_why})" if mode == "spectrum-mc" else ""))
    elif mode == "allgather":
        # every rank transforms 1/world of the step's blocks; ONE all-gather hands every block's spectrum to everybody
        # (each block is still broadcast exactly once -- by the rank that transformed it)
        if B % world:
            raise SystemExit("--mg-mode allgather needs blocks-per-step divisible by the number of GPUs")
        Bq = B // world

        def fwd_part(step, slot):
            cz.forward(d_stream, Bq, spec2[slot][rank * Bq:(rank + 1) * Bq], scale=w.scale,
                       first_block=(step % ngroups) * B + rank * Bq)

        sharder = PipelinedSharder(rank, world, forward=fwd_part, channels=chan, depth=nslots, forward_on_all=True,
                                   broadcast=lambda slot: dist.all_gather_into_tensor(
                                       spec2[slot].view(-1), spec2[slot][rank * Bq:(rank + 1) * Bq].reshape(-1), async_op=True))
        par = (f"{world} GPUs: every rank transforms {Bq} of the step's {B} blocks, 1 NCCL all-gather of the spectra per step")
    elif mode == "a2a":
        # block-parallel forward + slice hand-off: every rank transforms 1/world of the step's blocks and sends each peer only
        # the bins that peer's channels read (ONE all-to-all per step; cfg-5: 7 x 6 MB out of every rank instead of 363 MB in)
        if B % world:
            raise SystemExit("--mg-mode a2a needs blocks-per-step divisible by the number of GPUs")
        Bq = B // world
        from ka9q_radio_b200 import workloads
        lo_hi = []
        for r in range(world):
            wr = workloads.by_name(w.name, r, world)
            lo = max(0, min(abs(c.shift) for c in wr.channels) - 304) // 4 * 4
            lo_hi.append((lo, min(cz.master.bins, max(abs(c.shift) for c in wr.channels) + 304)))
        width = max(hi - lo for lo, hi in lo_hi)
        a_send = [torch.zeros((world, Bq, width), dtype=torch.complex64, device=dev) for _ in range(nslots)]
        a_recv = [torch.empty((world, Bq, width), dtype=torch.complex64, device=dev) for _ in range(nslots)]

        from ka9q_radio_b200.sharding import SliceExchange
        sx = SliceExchange(rank, world, lo_hi, cz.master.spec_stride, Bq)   # pack / unpack: one strided copy each when regular

        def fwd_part(step, slot):
            mine = spec2[slot][rank * Bq:(rank + 1) * Bq]
            cz.forward(d_stream, Bq, mine, scale=w.scale, first_block=(step % ngroups) * B + rank * Bq)
            sx.pack(mine, a_send[slot])

        def exchange(slot):
            h = dist.all_to_all_single(a_recv[slot].view(-1), a_send[slot].view(-1), async_op=True)
            return _Multi([h], then=lambda: sx.unpack(spec2[slot], a_recv[slot]))

        sharder = PipelinedSharder(rank, world, forward=fwd_part, channels=chan, depth=nslots, forward_on_all=True, broadcast=exchange)
        par = (f"{world} GPUs: every rank transforms {Bq} of the step's {B} blocks and sends each peer only the bins its channels "
               f"read ({(lo_hi[0][1] - lo_hi[0][0]) * 8 / 1e6:.2f} MB of {cz.master.bins * 8 / 1e6:.2f} MB per block), 1 NCCL all-to-all per step")
    elif mode == "slices":
        # slice hand-off: rank r only receives the bins its own channels read (cfg-5: 1024 x 188 + 600 bins of 1 620 001)
        lo_hi = [None] * world
        from ka9q_radio_b200 import workloads
        for r in range(world):
            wr = workloads.by_name(w.name, r, world)
            lo = max(0, min(abs(c.shift) for c in wr.channels) - 304) // 4 * 4
            hi = min(cz.master.bins, max(abs(c.shift) for c in wr.channels) + 304)
            lo_hi[r] = (lo, hi)

        width = max(hi - lo for lo, hi in lo_hi)
        stage = [torch.empty((world, B, width), dtype=torch.complex64, device=dev) if rank == 0 else None for _ in range(nslots)]
        recv = [torch.empty((B, width), dtype=torch.complex64, device=dev) for _ in range(nslots)]

        def hand_off(slot):
            # ONE scatter per step: rank 0 packs every rank's bin window into a staging tensor (a strided device copy)
            if rank == 0:
                for r in range(1, world):
                    lo, hi = lo_hi[r]
                    stage[slot][r, :, : hi - lo].copy_(spec2[slot][:, lo:hi])
                h = dist.scatter(recv[slot], [stage[slot][r] for r in range(world)], src=0, async_op=True)
                return h
            lo, hi = lo_hi[rank]
            h = dist.scatter(recv[slot], None, src=0, async_op=True)
            return _Multi([h], then=lambda: spec2[slot][:, lo:hi].copy_(recv[slot][:, : hi - lo]))

        sharder = PipelinedSharder(rank, world, forward=fwd, channels=chan, depth=nslots, broadcast=hand_off)
        par = (f"{world} GPUs: forward on rank 0, each rank receives only the bins its channels read "
               f"({(lo_hi[1][1] - lo_hi[1][0]) * 8 / 1e6:.2f} MB of {cz.master.bins * 8 / 1e6:.2f} MB per block), NCCL send/recv")
    else:
        # alternative (SURVEY.md 8e): broadcast the raw int16 window (half the bytes) and replicate
        # the forward transform on every GPU
        nwin = hist + B * wpb
        win2 = [torch.empty(nwin, dtype=torch.int16, device=dev) for _ in range(nslots)]

        def stage(step, slot):
            g = (step % ngroups) * B * wpb
            win2[slot].copy_(d_stream[g:g + nwin])

        def chan_after_forward(step, slot):
            cz.forward(win2[slot], B, spec2[slot], scale=w.scale)
            cz.channels(spec2[slot], B, out)

        sharder = PipelinedSharder(rank, world, forward=stage, channels=chan_after_forward, depth=nslots,
                                   broadcast=lambda slot: dist.broadcast(win2[slot].view(torch.uint8), src=0, async_op=True))
        par = f"{world} GPUs: 1 NCCL broadcast of the int16 window per step, forward replicated"

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sharder.run(range(args.warmup))
    barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # hold the same load for ~0.4 s before timing: clocks settle, and nvidia-smi (20 ms period) gets
    # samples under exactly this workload even when the K timed steps last only milliseconds
    nhold = max(args.warmup, int(0.4 / max(1e-4, 2.5e-5 * B)))
    sharder.run(range(nhold))
    barrier()
    lib.kgpu_profile_enable(1)
    lib.kgpu_profile_reset()
    launches0 = lib.kgpu_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(comp)
    sharder.run(range(args.warmup, args.warmup + args.steps))
    e1.record(comp)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = lib.kgpu_launch_count() - launches0
    prof = capi.profile_snapshot()
    lib.kgpu_profile_enable(0)
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    samples = args.steps * B * L
    stream_msps = samples / (ms * 1e-3) / 1e6
    value = stream_msps * world          # every rank runs the stream through its own 1024-channel bank

    # ---- parity of the configuration that was just timed: outputs of the LAST step vs the oracle --------------
    last_step = args.warmup + args.steps - 1
    fb = (last_step % ngroups) * B
    blocks_chk = sorted({0, B // 2 - 1 if B > 2 else 0, B - 1})
    stride = max(1, nchan // 22)
    chans_chk = sorted(set(list(range(0, nchan, stride)) + [nchan - 1] + _tone_channels(w)))
    o_host = out.cpu().numpy()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w, cz, o_host)
    pairs = {}
    for b in blocks_chk:
        for c in chans_chk:
            off = cz.bank.out_offset(c)
            pairs[(b, c)] = np.ascontiguousarray(o_host[b, off: off + w.channels[c].olen])
    parity = parity_check(w, host, pairs, fb) if not args.quick else {"max_rel_err": None, "checked": 0, "skipped": "--quick"}
    if world > 1:   # every rank checks its own bank; rank 0 reports the worst
        v = torch.tensor([parity["max_rel_err"] if parity.get("max_rel_err") is not None else 1.0, float(parity.get("checked", 0))],
                         dtype=torch.float64, device=dev)
        vmax = v.clone()
        dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
        vsum = v.clone()
        dist.all_reduce(vsum, op=dist.ReduceOp.SUM)
        parity["max_rel_err"] = float(vmax[0].item())
        parity["checked"] = int(vsum[1].item())
        parity["ok"] = parity["max_rel_err"] < 1e-5
        parity["ranks"] = world

    # ---- end to end through the C-ABI with HOST buffers (pinned), copies inside the timed region
    e2e = run_e2e(args, torch, cz, hpin, dev, rank, world, dist, B, ngroups, w, hist) if not args.quick else {"value": 0.0, "skipped": "--quick"}
    if rank == 0 and world == 1 and not args.no_filter_h and not args.quick:
        cz_state = None
        try:
            e2e["filter_h"] = run_e2e_filter_h(args, w, host)
        except Exception as ex:  # the kgpu-level e2e stands on its own
            e2e["filter_h"] = {"error": str(ex)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel, from the per-launch CUDA-event times ---------------
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "6650 GB/s (of fallback, B200_PROFILING.md)"
    blocks_fwd = B // world if mode in ("allgather", "a2a") else B
    alg_per_kernel = {"fwd_cols": alg_fwd_in * blocks_fwd, "fwd_rows": alg_fwd_out * blocks_fwd, "chan": alg_chan * B}
    kernels = {}
    for name, (tot_ms, cnt) in prof.items():
        if cnt:
            avg = tot_ms / cnt
            per_step = tot_ms / args.steps
            kernels[name] = {"launches": cnt, "avg_ms": avg, "ms_per_step": per_step,
                             "alg_bytes_per_step": alg_per_kernel.get(name, 0.0),
                             "alg_gbs": alg_per_kernel.get(name, 0.0) / (per_step * 1e-3) / 1e9 if per_step > 0 else None}
    cand = {k: v for k, v in kernels.items() if k in alg_per_kernel}
    dom = max(cand, key=lambda k: cand[k]["ms_per_step"]) if cand else None
    traffic = TRAFFIC_NCU.get(w.name, TRAFFIC_NCU if w.name == "cfg2" else {})
    roof = None
    if dom:
        a = kernels[dom]["alg_gbs"]
        tr = traffic.get(dom) if isinstance(traffic, dict) else None
        roof = {"kernel": dom, "bound": "hbm", "achieved": a, "peak": peak, "unit": "GB/s", "frac": a / peak,
                "traffic": (tr * blocks_fwd if dom != "chan" else tr * B) if isinstance(tr, (int, float)) else None,
                "traffic_note": "ncu dram__bytes_read+write per block (profiles/traffic.json) x blocks per step",
                "peak_source": peak_src,
                "note": "algorithmic bytes attributed per kernel: fwd_cols = window read, fwd_rows = spectrum "
                        "write (bins*8 B), chan = slices+responses+outputs; the inter-pass buffer earns no credit"}
    sum_ms = sum(v["ms_per_step"] for k, v in kernels.items() if k in alg_per_kernel)
    pipeline = {"alg_bytes_per_step": alg_bytes * B, "kernel_ms_per_step": sum_ms,
                "achieved": alg_bytes * B / (sum_ms * 1e-3) / 1e9 if sum_ms else None, "unit": "GB/s"}
    if pipeline["achieved"]:
        pipeline["frac"] = pipeline["achieved"] / peak
    pipeline["achieved_wall"] = alg_bytes * B * args.steps / (ms * 1e-3) / 1e9
    pipeline["frac_wall"] = pipeline["achieved_wall"] / peak

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_reference_run(w.name, blocks=args.ref_blocks, steps=2, warmup=1)["cpu_baseline"]
        except Exception as ex:  # the GPU numbers stand on their own
            cpu = {"value": None, "unit": "Msamples/s", "cores": os.cpu_count(), "kind": "reference", "sample": f"failed: {ex}"}

    line = {
        "metric": METRIC, "value": value, "unit": "Msamples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w.description + (" per GPU" if world > 1 else ""),
                   "blocks_per_step": B, "input_stream_MB": round(host.nbytes / 1e6, 1),
                   "l2_policy": f"input stream larger than L2 (126 MB) -- this rank cycles through {rank_reads * (nstream // B) / 1e6:.0f} MB "
                                "of it --, consecutive groups cycled; no explicit flush",
                   "plan": cz.master.describe(), "parallelism": par,
                   "value_definition": ("input stream rate" if world == 1 else
                                        "channel-weighted: stream rate x GPUs (every GPU runs the whole sample stream through its own "
                                        f"{nchan}-channel bank); the single-stream input rate is config.stream_msps"),
                   "stream_msps": stream_msps, "realtime_factor": stream_msps / (w.fs / 1e6)},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "roofline": roof,
        "roofline_pipeline": pipeline, "kernels": kernels, "parity": parity, "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64_000_000


def dump_outputs(dirname: str, w, cz, o_host: np.ndarray) -> None:
    """The channel outputs of the last timed step as a caller of the channel bank receives them: for each block of the step,
    every channel's olen complex samples in channel order -> DIR/outputs.npy, float32 [blocks, samples, 2] (re, im).
    Outputs larger than DUMP_BYTES (all files together) are sampled with a fixed seed: whole blocks, and whole channels
    only when one block alone is too large.  DIR/blocks.npy and DIR/channels.npy list what was kept (float64 indices within
    the step and the workload's channel list).  With several GPUs these are rank 0's channels."""
    rng = np.random.default_rng(0)
    nb, n = o_host.shape[0], len(w.channels)
    olen = np.array([c.olen for c in w.channels])
    budget = DUMP_BYTES - 8 * (nb + n) - 3 * 128          # the two index files and the three .npy headers
    chans = np.arange(n)
    if olen.sum() * 8 > budget:
        order = rng.permutation(n)
        chans = np.sort(order[: np.searchsorted(np.cumsum(olen[order]) * 8, budget, side="right")])
        if chans.size == 0:
            raise SystemExit(f"--dump-outputs: one channel's block alone exceeds {DUMP_BYTES} bytes")
    idx = np.concatenate([np.arange(cz.bank.out_offset(c), cz.bank.out_offset(c) + olen[c]) for c in chans])
    keep = min(nb, budget // (idx.size * 8))
    blocks = np.arange(nb) if keep == nb else np.sort(rng.choice(nb, keep, replace=False))
    outs = np.ascontiguousarray(o_host[np.ix_(blocks, idx)]).view(np.float32).reshape(len(blocks), idx.size, 2)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "outputs.npy"), outs)
    np.save(os.path.join(dirname, "blocks.npy"), blocks.astype(np.float64))
    np.save(os.path.join(dirname, "channels.npy"), chans.astype(np.float64))


class _Multi:
    """several async Work handles behind one .wait(), plus an optional completion action"""

    def __init__(self, hs, then=None):
        self.hs, self.then = hs, then

    def wait(self):
        for h in self.hs:
            h.wait()
        if self.then:
            self.then()


# ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per block and kernel (filled from profiles/ once captured)
TRAFFIC_NCU: dict = {}
try:
    TRAFFIC_NCU = json.loads((ROOT / "profiles" / "traffic.json").read_text())
except Exception:
    pass


def run_e2e(args, torch, cz, hpin, dev, rank, world, dist, B, ngroups, w, hist) -> dict:
    """Same metric through the C-ABI with HOST buffers: every step copies that step's window
    (M-1 history + B*L new int16 samples) from pinned host memory, runs forward + channels and
    reads the channel outputs back into pinned host memory.  Copies are double-buffered on
    separate streams (a streaming receiver would do the same); all of it is inside the timed region."""
    wpb = w.samples_per_block
    nwin = hist + B * wpb
    d_in = [torch.empty(nwin, dtype=torch.int16, device=dev) for _ in range(2)]
    d_out = [cz.alloc_outputs(B) for _ in range(2)]
    d_spec = [cz.alloc_spectra(B) for _ in range(2)]
    h_out = [torch.empty(d_out[0].shape, dtype=torch.complex64).pin_memory() for _ in range(2)]
    s_in, s_comp, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]
    steps, warm = args.steps, args.warmup

    def one(s):
        j = s & 1
        g = s % ngroups
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_comp[j])               # previous use of d_in[j] finished
            d_in[j].copy_(hpin[g * B * wpb: g * B * wpb + nwin], non_blocking=True)
            ev_in[j].record(s_in)
        with torch.cuda.stream(s_comp):
            s_comp.wait_event(ev_in[j])
            s_comp.wait_event(ev_out[j])              # previous D2H of d_out[j] finished
            if rank == 0 or world == 1:
                cz.forward(d_in[j], B, d_spec[j], scale=w.scale)
            if world > 1:
                dist.broadcast(d_spec[j], src=0)
            cz.channels(d_spec[j], B, d_out[j])
            ev_comp[j].record(s_comp)
        with torch.cuda.stream(s_out):
            s_out.wait_event(ev_comp[j])
            h_out[j].copy_(d_out[j], non_blocking=True)
            ev_out[j].record(s_out)

    for s in range(warm):
        one(s)
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize(dev)
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record(s_in)
    for s in range(steps):
        one(warm + s)
    s_out.synchronize()
    s_comp.synchronize()
    t1.record(s_out)
    torch.cuda.synchronize(dev)
    ms = t0.elapsed_time(t1)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    v = steps * B * w.L / (ms * 1e-3) / 1e6 * world
    return {"value": v, "unit": "Msamples/s", "h2d_bytes_per_step": int(nwin * 2),
            "d2h_bytes_per_step": int(d_out[0].numel() * 8), "ms_per_step": ms / steps,
            "api": "kgpu_forward + kgpu_bank_run (C-ABI, include/ka9q_gpu.h) on pinned host buffers, "
                   "H2D/compute/D2H double-buffered on 3 streams"}


def run_e2e_filter_h(args, w, host: np.ndarray) -> dict:
    """The drop-in path itself: pinned-or-not HOST int16 -> write_i16filter -> execute_filter_output_batch for every
    slave, through libka9qgpu.so's filter.h symbols only (tools/filterh_bench.c drives them from a producer and a
    consumer thread, as radiod's USB callback and channel threads would).  Parity of the last block vs the oracle."""
    so = ROOT / "tools" / "_build" / "filterh_bench.so"
    if not so.exists():
        raise RuntimeError("tools/_build/filterh_bench.so not built (python -c 'import __graft_entry__ as g; g.build()')")
    os.environ.setdefault("KA9Q_GPU_SPECTRUM_D2H", "0")   # noise is estimated on the device; nothing reads fdomain[] here
    os.environ.setdefault("KA9Q_GPU_ZEROCOPY", "1")
    H = C.CDLL(str(so))
    n = len(w.channels)
    ia = lambda xs: (C.c_int * n)(*xs)
    da = lambda xs: (C.c_double * n)(*xs)
    H.kgf_e2e_run.restype = C.c_double
    H.kgf_e2e_run.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_int,
                              C.POINTER(C.c_long), C.c_void_p, C.POINTER(C.c_uint), C.c_int]
    max_olen = max(c.olen for c in w.channels)
    chk = np.zeros((n, max_olen), np.complex64)
    last = C.c_long(0)
    lat = (C.c_double * 2)()
    drops = C.c_uint(0)
    k = args.filter_h_blocks_per_write
    nblk = args.filter_h_blocks
    stream_blocks = len(host) // w.samples_per_block
    def run(inplace):
        s = H.kgf_e2e_run(w.L, w.M, w.in_type, n, C.cast(ia([c.olen for c in w.channels]), C.c_void_p),
                          C.cast(ia([c.shift for c in w.channels]), C.c_void_p), C.cast(da([c.low for c in w.channels]), C.c_void_p),
                          C.cast(da([c.high for c in w.channels]), C.c_void_p), C.cast(da([c.beta for c in w.channels]), C.c_void_p),
                          host.ctypes.data, stream_blocks, k, 8, nblk, w.scale, chk.ctypes.data, max_olen, C.byref(last),
                          C.cast(lat, C.c_void_p), C.byref(drops), inplace)
        if s <= 0:
            raise RuntimeError(f"kgf_e2e_run failed ({s})")
        return s

    secs_copy = run(0)     # write_i16filter(samples): CPU memcpy of every sample into the pinned ring, then H2D
    copy_msps = nblk * w.L / secs_copy / 1e6
    H.kgf_ring_words.restype = C.c_long
    ring_words = H.kgf_ring_words(w.L, w.M, w.in_type)
    wpb = w.samples_per_block
    ring_src = np.ascontiguousarray(w.stream(ring_words // wpb + 2)[:ring_words])
    host_keep, host = host, ring_src          # run() reads `host`
    stream_blocks = ring_words // wpb + 2
    secs = run(1)          # samples already in the pinned ring (a driver's DMA target): publish only
    host = host_keep
    msps = nblk * w.L / secs / 1e6
    res = {"value": msps, "unit": "Msamples/s", "realtime_factor": msps / (w.fs / 1e6), "blocks": nblk, "blocks_per_write": k,
           "ms_per_block": 1e3 * secs / nblk, "latency_ms_mean": lat[0], "latency_ms_max": lat[1], "dropped_blocks": int(drops.value),
           "with_ring_memcpy": {"value": copy_msps, "unit": "Msamples/s", "realtime_factor": copy_msps / (w.fs / 1e6),
                                "note": "same leg with write_i16filter(samples) copying every sample from a pageable host buffer into the ring first"},
           "ingest": "samples deposited in the library's pinned ring (filter_i16_write_pointer: the DMA target a patched rx888.c:797-826 "
                     "would hand libusb), published with write_i16filter(NULL, n)",
           "slaves": n, "h2d_bytes_per_block": int((w.samples_per_block + (w.M - 1) * (2 if w.in_type == 1 else 1) / k) * 2),
           "d2h_bytes_per_block": int(sum(c.olen for c in w.channels) * 8),
           "api": "create_filter_input/create_filter_output/set_filter/write_i16filter/execute_filter_output_batch "
                  "(filter.h surface of libka9qgpu.so), host int16 in, host complex out, zero-copy delivery, "
                  f"{k} blocks per write_i16filter call"}
    start = int(last.value)   # word index of the last block's window inside the cyclic ring contents
    nwin = wpb + (w.M - 1) * (2 if w.in_type == 1 else 1)
    window = ring_src[(start + np.arange(nwin)) % ring_words]
    stride = max(1, n // 22)
    chans = sorted(set(list(range(0, n, stride)) + [n - 1] + _tone_channels(w)))
    pairs = {(0, c): np.ascontiguousarray(chk[c, : w.channels[c].olen]) for c in chans}
    res["parity"] = parity_check(w, host, pairs, 0, windows={0: window})
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configuration (default: cfg2 on one GPU, cfg5's channel plan on several)")
    ap.add_argument("--blocks-per-step", type=int, default=32)
    ap.add_argument("--stream-blocks", type=int, default=64, help="resident input stream length (blocks)")
    ap.add_argument("--ref-blocks", type=int, default=12, help="blocks per step of the CPU reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-filter-h", action="store_true", help="skip the e2e leg through the filter.h symbols")
    ap.add_argument("--filter-h-blocks", type=int, default=96)
    ap.add_argument("--filter-h-blocks-per-write", type=int, default=1,
                    help="blocks completed per write_i16filter call (1..ND-1); 1 keeps ND launches in flight: 13.7 GS/s against 7.9-9.1 (2) and 10.0 (3)")
    ap.add_argument("--quick", action="store_true", help="sweeps: skip the parity self-check and the e2e legs")
    ap.add_argument("--depth", type=int, default=2, help="spectrum ring depth of the multi-GPU pipeline")
    ap.add_argument("--mg-mode", default="a2a", choices=["spectrum", "spectrum-mc", "input", "allgather", "slices", "a2a"],
                    help="multi-GPU hand-off of the shared forward spectrum, one NCCL collective per step: `allgather` (default) = every "
                         "rank transforms 1/N of the step's blocks and each block's spectrum is broadcast once by the rank that made it; "
                         "`spectrum` = all blocks transformed on rank 0 + one ncclBroadcast (north_star's literal form: rank 0's NVLink "
                         "egress and HBM bound it); `spectrum-mc` = the same through this repository's NVSwitch-multicast copy kernel; "
                         "`input` = broadcast of the raw window, forward replicated; `slices` = rank 0 scatters per-rank bin slices; "
                         "`a2a` = block-parallel forward + all-to-all of per-rank bin slices")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="GPU arm: write the channel outputs of the last timed step to DIR/outputs.npy (float32, at most "
                         "64 MB: a fixed sample of the step's blocks when larger; DIR/blocks.npy and DIR/channels.npy list them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; the reference arm only times")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
