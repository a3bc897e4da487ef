"""The C-ABI library loads without a GPU and exports every symbol include/pamg.h declares."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from parallel_amg_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "pamg.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(pamg_[a-z_0-9]+)\s*\(", txt)))


def test_header_symbols_exported_and_bound():
    lib = L.load()
    names = declared_symbols()
    assert len(names) >= 40
    for n in names:
        assert hasattr(lib, n), f"{n} declared in pamg.h but not exported by libpamg.so"
        assert n in L.PROTOTYPES, f"{n} has no ctypes prototype"
    assert set(L.PROTOTYPES) == set(names)


def test_struct_sizes_match_c_layout():
    lib = L.load()
    o = L.Options()
    lib.pamg_default_options(C.byref(o))
    assert o.struct_size == C.sizeof(L.Options)
    assert (o.coarse_size, o.nu_pre, o.nu_post, o.use_graph) == (500, 1, 1, 1)
    assert abs(o.omega_jacobi - 2.0 / 3.0) < 1e-16


def test_device_calls_fail_loudly_without_init():
    c = L.Context(1)
    c.gallery_poisson((8, 8), (1, 1))
    c.setup()
    c.local_parts = [0]
    with pytest.raises(L.PamgError) as e:
        c.spmv(0, [np.zeros(64)])
    assert e.value.status == L.ERR_ARG and "device not initialised" in str(e.value)


def _gpu_visible():
    # ask CUDA rather than look for a device node: a container may expose its GPU under another /dev name
    try:
        import torch
        return torch.cuda.device_count() > 0
    except Exception:
        return False


@pytest.mark.skipif(_gpu_visible(), reason="GPU present")
def test_no_gpu_is_an_error_not_a_fallback():
    c = L.Context(1)
    c.gallery_poisson((8, 8), (1, 1))
    c.setup()
    with pytest.raises(L.PamgError) as e:
        c.device_init()
    assert e.value.status in (L.ERR_NOGPU, L.ERR_CUDA)
