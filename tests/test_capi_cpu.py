"""CPU suite (no GPU): the C-ABI library loads and exports every symbol include/*.h declares;
the pure-host planner makes sane choices.  No compute entry point is called here."""
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def test_library_exports_every_declared_symbol():
    from ka9q_radio_b200 import capi

    lib = capi.load()
    syms = capi.exported_symbols()
    assert len(syms) >= 25
    missing = [s for s in syms if not hasattr(lib, s)]
    assert not missing, missing


def test_filter_abi_symbols_exported():
    """The reference-facing surface (filter.h:99-118) must be exported by the same library."""
    import ctypes

    from ka9q_radio_b200 import capi

    hdr = (ROOT / "include" / "ka9q_gpu_filter.h")
    if not hdr.exists():
        pytest.skip("filter.h layer not built yet")
    lib = capi.load()
    names = set(re.findall(r"\b([a-z_0-9]+)\s*\(", hdr.read_text()))
    wanted = {"create_filter_input", "create_filter_output", "execute_filter_input", "execute_filter_output",
              "delete_filter_input", "delete_filter_output", "set_filter", "set_filter_weights", "write_cfilter",
              "write_rfilter", "write_i16filter"}
    assert wanted <= names
    for n in wanted:
        assert hasattr(lib, n), n


@pytest.mark.parametrize("n,maxstages", [(600, 2), (300, 2), (1200, 3), (1296, 3), (1250, 3), (625, 2), (2048, 3), (30000 // 150, 2)])
def test_planner_radices(n, maxstages):
    from ka9q_radio_b200 import capi

    r = capi.plan_radices(n)
    prod = 1
    for v in r:
        prod *= v
    assert prod == n and len(r) <= maxstages
    # even radices precede odd ones (unit-stride stages stay bank-conflict free)
    seen_odd = False
    for v in r:
        if v % 2:
            seen_odd = True
        else:
            assert not seen_odd


def test_planner_rejects_large_primes():
    from ka9q_radio_b200 import capi

    with pytest.raises(capi.KgpuError):
        capi.plan_radices(2 * 19)


@pytest.mark.parametrize("n", [1620000, 30000, 500000, 3000, 250000])
def test_planner_split(n):
    from ka9q_radio_b200 import capi

    a, b = capi.plan_split(n)
    assert a * b == n and a >= b and a <= 4096


def test_no_oracle_in_product():
    """The shipped package must not import, link or call anything under oracle/."""
    pkg = ROOT / "ka9q_radio_b200"
    for p in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")) + list(pkg.rglob("*.c")) + list(pkg.rglob("Makefile")):
        txt = p.read_text()
        assert "oracle" not in txt.replace("no oracle", ""), p


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the driver's reference arm) times oracle/_ref (or the port) on the
    host cores and prints the contract's JSON line; no GPU involved."""
    import json
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    if not (root / "oracle" / "_ref" / "libka9qref.so").exists():
        pytest.skip("oracle/_ref is built only where the reference's sources are readable")
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--ref-blocks", "2"], capture_output=True, text=True, timeout=600, check=True)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "Msamples/s" and line["value"] > 0
    assert line["e2e"]["value"] == line["value"] and line["e2e"]["h2d_bytes_per_step"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and "sample" in cb


def test_butterfly_templates_on_host(tmp_path):
    """fft_radix.cuh compiled for the HOST (the packed f32x2 primitives fall back to scalar code with the same
    rounding): every radix the planner can pick, forward and inverse, against a float64 DFT."""
    import shutil
    import subprocess
    from pathlib import Path

    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not Path(nvcc).exists():
        pytest.skip("nvcc not available")
    src = Path(__file__).resolve().parent / "host" / "dft_host_test.cu"
    exe = tmp_path / "dft_host_test"
    subprocess.run([nvcc, "-std=c++17", "-O1", "--expt-relaxed-constexpr", "-gencode", "arch=compute_100a,code=sm_100a",
                    "-o", str(exe), str(src)], check=True, capture_output=True, timeout=600)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert out.returncode == 0 and "all butterflies ok" in out.stdout, out.stdout[-2000:]
