"""GPU: drop-in acceptance with the reference's OWN drivers.  oracle/Makefile compiles the unmodified
dctz-test.c (both build modes, Makefile:12-17) and dct-test.c (its line 16) of the DCTZ sources named by REF against the
reference's own headers and links them against libdctz_ec.so / libdctz_qt.so instead of the reference's sources
(oracle/_ref/dropin-*).  They must behave like the all-reference binaries built from the same drivers
(oracle/_ref/dctz-{ec,qt}-test, dct-test): same files, same summary lines, the same reconstruction to DCT tolerance.
The repository does not contain the reference sources: without them these comparisons skip.  The library's debug
output is checked through the project's own driver (dctz-ec-test, the reference driver's command line)."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from dctz_b200 import fields

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")
BIN = os.path.join(ROOT, "dctz_b200", "bin")


def _need(*names):
    missing = [n for n in names if not os.path.exists(os.path.join(REF, n))]
    if missing:
        pytest.skip(f"oracle/_ref lacks {missing}: they are built from the unmodified DCTZ sources (make -C oracle REF=<dir>)")


def _run(binary, args, cwd, env=None, where=REF):
    p = subprocess.run([os.path.join(where, binary), *args], cwd=cwd, capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, **(env or {})))
    assert p.returncode == 0, f"{binary} failed ({p.returncode}):\n{p.stdout[-2000:]}\n{p.stderr[-2000:]}"
    return p.stdout


def _summary(txt):
    m = re.search(r"CR = ([0-9.]+), PSNR = ([0-9.infa-]+)", txt)
    assert m, txt[-1500:]
    return float(m.group(1)), float(m.group(2))


@pytest.mark.parametrize("mode,flag,dtype,dims", [("ec", "-d", np.float64, ("3600", "1800")), ("qt", "-f", np.float32, ("3600", "1800")),
                                                 ("ec", "-f", np.float32, ("64", "1000", "7")), ("qt", "-d", np.float64, ("229",))])
def test_reference_driver_linked_against_the_drop_in(tmp_path, mode, flag, dtype, dims):
    """dctz-test.c:181,250 -> dctz_compress / dctz_decompress / calc_psnr of libdctz_{ec,qt}.so; configs[0] and
    configs[1] shapes plus a 3-D float case and a tiny one with a ragged tail block."""
    _need(f"dropin-{mode}-test", f"dctz-{mode}-test")
    n = int(np.prod([int(d) for d in dims]))
    x = fields.cesm_like(dtype=dtype)[:n] if n > 229 else fields.small_cases(dtype)["three_blocks_tail37"]
    outs = {}
    for who, binary in (("ours", f"dropin-{mode}-test"), ("ref", f"dctz-{mode}-test")):
        d = tmp_path / who
        d.mkdir()
        x.tofile(d / "f.bin")
        txt = _run(binary, [flag, "1E-3", "var", "f.bin", *dims], str(d))
        assert f"total number of elements = {n}" in txt and "outSize = " in txt and txt.rstrip().endswith("done")
        z = np.fromfile(d / f"f.bin.{mode}.1E-3.z", dtype=np.uint8)
        r = np.fromfile(d / f"f.bin.{mode}.1E-3.z.r", dtype=dtype)
        side = sorted(p.name for p in d.iterdir())
        outs[who] = dict(txt=txt, z=z, r=r, side=side, cr_psnr=_summary(txt))
    assert outs["ours"]["side"] == outs["ref"]["side"]  # bin_index.bin, AC_exact.bin (+ qtable.bin), .z, .z.r
    ours, ref = outs["ours"], outs["ref"]
    tol = (1e-12 if dtype == np.float64 else 1e-5) * 8 * float(np.max(np.abs(x)))
    assert ours["r"].size == n and float(np.max(np.abs(ours["r"].astype(np.float64) - ref["r"].astype(np.float64)))) <= tol
    assert abs(int(ours["z"].size) - int(ref["z"].size)) <= max(64, ref["z"].size // 200)  # the chunk-parallel deflate adds a few bytes per MiB
    assert abs(ours["cr_psnr"][0] - ref["cr_psnr"][0]) <= 0.02 * ref["cr_psnr"][0] and abs(ours["cr_psnr"][1] - ref["cr_psnr"][1]) <= 0.01
    # header fields (dctz.h:96-119); padding bytes and the unused halves of the float unions are not compared (the
    # reference leaves them uninitialised), the mean is order dependent, the section sizes depend on the deflate chunking
    from tests import reflib

    ho = np.frombuffer(ours["z"][:56].tobytes(), dtype=reflib.HEADER_DTYPE)[0]
    hr = np.frombuffer(ref["z"][:56].tobytes(), dtype=reflib.HEADER_DTYPE)[0]
    for key in ("datatype", "num_elements", "error_bound"):
        assert ho[key] == hr[key], key
    assert abs(int(ho["tot_AC_exact_count"]) - int(hr["tot_AC_exact_count"])) <= 8  # ties only
    es = np.dtype(dtype).itemsize
    assert ho["scaling_factor"].tobytes()[:es] == hr["scaling_factor"].tobytes()[:es]
    mo, mr = (np.frombuffer(h["mean"].tobytes()[:es], dtype=dtype)[0] for h in (ho, hr))
    assert abs(float(mo) - float(mr)) <= (1e-9 if dtype == np.float64 else 1e-3) * max(1.0, abs(float(mr)))
    if mode == "qt":
        assert ho["bindex_count"] == hr["bindex_count"] == n


def test_reference_driver_time_debug_lines_and_dct_dumps(tmp_path):
    """DCTZ_TIME_DEBUG=1 prints the reference's -DTIME_DEBUG stage lines (dctz-comp-lib.c:762-773, dctz-decomp-lib.c:513-528)
    with CUDA-event stage times; DCTZ_DCT_FILE_DEBUG=1 writes dct_result.bin / DC.bin like -DDCT_FILE_DEBUG (:422-433)."""
    x = fields.cesm_like()[:64 * 4000 + 21]
    x.tofile(tmp_path / "f.bin")
    txt = _run("dctz-ec-test", ["-d", "1E-3", "var", "f.bin", str(x.size)], str(tmp_path), env=dict(DCTZ_TIME_DEBUG="1", DCTZ_DCT_FILE_DEBUG="1"),
               where=BIN)
    assert re.search(r"sf_t=[0-9.]+\(s\), dct_t=[0-9.]+\(s\), zlib_t\(compress\)=[0-9.]+\(s\)", txt), txt
    assert re.search(r"sf_t=[0-9.]+\(s\), idct_t=[0-9.]+\(s\), zlib_t\(uncompress\)=[0-9.]+\(s\)", txt), txt
    assert "comp_time = " in txt and "decomp_time = " in txt
    from tests import reflib

    coef = np.fromfile(tmp_path / "dct_result.bin", dtype=np.float64)
    dc = np.fromfile(tmp_path / "DC.bin", dtype=np.float32)
    o = reflib.oracle_compress(x, 1e-3, False)
    assert coef.size == x.size and dc.size == (x.size + 63) // 64
    assert float(np.max(np.abs(coef - o["coef"]))) <= 1e-12 * float(np.max(np.abs(o["coef"]))) * 4
    assert np.allclose(dc, o["dc"], rtol=2e-7, atol=0)


@pytest.mark.parametrize("flag,dtype", [("-d", np.float64), ("-f", np.float32)])
def test_reference_dct_test_linked_against_the_drop_in(tmp_path, flag, dtype):
    """dct-test.c: dct_init / dct_fftw / ifft_idct / dct_finish (dct.h:17-27), one block per call, incl. the odd tail."""
    _need("dropin-dct-test", "dct-test")
    rng = np.random.default_rng(12)
    n = 64 * 40 + 37
    x = (rng.standard_normal(n) * 3 + 1).astype(dtype)
    res = {}
    for who, binary in (("ours", "dropin-dct-test"), ("ref", "dct-test")):
        d = tmp_path / who
        d.mkdir()
        x.tofile(d / "f.bin")
        txt = _run(binary, [flag, "f.bin", str(n)], str(d))
        assert f"nblk={(n + 63) // 64}, rem={n % 64}" in txt
        res[who] = (np.fromfile(d / "f.bin.x", dtype=dtype).astype(np.float64), np.fromfile(d / "f.bin.r", dtype=dtype).astype(np.float64))
    tol = 1e-12 if dtype == np.float64 else 1e-5
    scale = float(np.max(np.abs(res["ref"][0])))
    assert float(np.max(np.abs(res["ours"][0] - res["ref"][0]))) <= tol * scale  # coefficients (f.bin.x)
    assert float(np.max(np.abs(res["ours"][1] - x.astype(np.float64)))) <= tol * scale * 4  # reconstruction (f.bin.r)
