"""CPU: the C-ABI libraries load and export every symbol their headers declare; without a GPU every
compute entry point fails loudly (there is no CPU fallback to fall into)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import dctz_b200
from dctz_b200 import binding

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared(header):
    txt = open(os.path.join(ROOT, "include", header)).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b([a-z_0-9]+)\s*\(", txt)) - {"defined", "sizeof"})


def test_gpu_header_symbols_are_exported():
    names = [n for n in _declared("dctz_gpu.h") if n.startswith("dctz_gpu_")]
    assert sorted(names) == sorted(binding.EXPORTS), set(names) ^ set(binding.EXPORTS)
    lib = dctz_b200.load_library()
    for n in names:
        assert hasattr(lib, n), n


@pytest.mark.parametrize("flavour", ["ec", "qt"])
def test_host_library_exports_the_reference_api(flavour):
    path = os.path.join(ROOT, "dctz_b200", f"libdctz_{flavour}.so")
    assert os.path.exists(path), "run __graft_entry__.build()"
    lib = C.CDLL(path)
    want = [n for n in _declared("dctz_compat.h") if not n.startswith("dctz_num")]
    for n in want:  # dctz.h:121-128 and dct.h:17-27
        assert hasattr(lib, n), n
    assert lib.dctz_build_is_qt() == (1 if flavour == "qt" else 0)


def test_no_cpu_fallback():
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is what the CPU box checks")
    lib = dctz_b200.load_library()
    assert lib.dctz_gpu_device_count() == 0
    with pytest.raises(dctz_b200.DctzGpuError) as e:
        dctz_b200.Context(0)
    assert e.value.code == -1  # DCTZ_GPU_ENODEV
    assert "no CUDA device" in str(e.value)


def test_info_struct_layout():
    assert binding.INFO_BYTES == 80  # 5 doubles + 4 u64 + 2 i32, mirrored by a static_assert in dctz_gpu.cu


def test_plan_struct_mirrors_the_header():
    """binding.LaunchPlan lists the fields of dctz_gpu_plan in the header's order (all uint64_t)"""
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "dctz_gpu.h")).read(), flags=re.S)
    body = re.search(r"typedef struct dctz_gpu_plan \{(.*?)\} dctz_gpu_plan;", txt, flags=re.S).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if decl:
            assert decl.startswith("uint64_t "), decl
            fields += [f.strip() for f in decl[len("uint64_t "):].split(",")]
    assert fields == [k for k, _ in binding.LaunchPlan._fields_]
    assert C.sizeof(binding.LaunchPlan) == 8 * len(fields)


def test_product_does_not_touch_the_oracle():
    """nothing under dctz_b200/ or include/ may import, link or call oracle/ (it is test infrastructure)."""
    bad = []
    for base in ("dctz_b200", "include"):
        for d, _, fs in os.walk(os.path.join(ROOT, base)):
            for f in fs:
                if f.endswith((".py", ".c", ".cu", ".cuh", ".h", "Makefile")):
                    txt = open(os.path.join(d, f), errors="ignore").read()
                    if re.search(r"liboracle|oracle_|from tests|import tests|oracle/", txt):
                        bad.append(os.path.join(d, f))
    assert not bad, bad
