"""CPU: the C-ABI library loads, exports every symbol include/dbslmm_b200.h declares, refuses to
run without a GPU (no fallback), and the host-only block scheduler behaves."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from dbslmm_b200 import _abi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    txt = open(os.path.join(ROOT, "include", "dbslmm_b200.h")).read()
    return sorted(set(re.findall(r"DBSLMM_B200_API\s+[\w\s\*]+?\b(dbslmm_b200_\w+)\s*\(", txt)))


def test_library_matches_the_header_exports_and_abi_version():
    lib = _abi.load()
    names = header_functions()
    assert len(names) >= 13
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_abi.EXPORTS) == names
    assert lib.dbslmm_b200_abi_version() == 6


def test_fit_args_struct_layout_matches_header():
    # natural alignment on LP64: the ctypes mirror must have the size of the C struct (17 + 7 + 3 + 1 fields)
    assert C.sizeof(_abi.FitArgs) == 216
    assert C.sizeof(_abi.Timing) == 88


def test_no_cpu_fallback():
    lib = _abi.load()
    if lib.dbslmm_b200_device_count() > 0:
        pytest.skip("a GPU is visible")
    h = C.c_void_p()
    assert lib.dbslmm_b200_create(0, C.byref(h)) == -1          # DBSLMM_B200_ERR_CUDA
    with pytest.raises(_abi.EngineError):
        _abi.Engine(0)


def _plan(m_s, m_l, n_ref, n_ranks):
    lib = _abi.load()
    m_s = np.ascontiguousarray(m_s, np.int32)
    owner = np.zeros(m_s.size, np.int32)
    cost = np.zeros(n_ranks)
    ml = None if m_l is None else np.ascontiguousarray(m_l, np.int32)
    rc = lib.dbslmm_b200_plan_shards(m_s.size, m_s.ctypes.data, None if ml is None else ml.ctypes.data, n_ref, n_ranks,
                                     owner.ctypes.data, cost.ctypes.data)
    assert rc == 0
    return owner, cost


def test_plan_shards_lpt_balance():
    from dbslmm_b200 import synth
    sizes = synth.eur_block_sizes(1_100_000, 3000)
    assert sizes.size == 1703 and sizes.max() <= 3000
    for g in (1, 2, 4, 8):
        owner, cost = _plan(sizes, None, 2000, g)
        assert owner.min() == 0 and owner.max() == g - 1
        assert np.bincount(owner, minlength=g).sum() == sizes.size
        assert cost.max() / cost.mean() < 1.02                      # LPT keeps the makespan within 2 % of the mean
    owner, _ = _plan([0, 0, 5], [0, 1, 0], 100, 2)
    assert set(owner.tolist()) <= {0, 1}


def test_plan_shards_rejects_bad_arguments():
    lib = _abi.load()
    assert lib.dbslmm_b200_plan_shards(3, None, None, 100, 2, None, None) == -2


def test_fit_args_field_offsets_match_the_c_header(tmp_path):
    """Field-by-field: offsetof() from a C program compiled against include/dbslmm_b200.h vs the ctypes mirror."""
    import subprocess
    fields = [name for name, _ in _abi.FitArgs._fields_]
    tfields = [name for name, _ in _abi.Timing._fields_]
    src = ['#include <stdio.h>', '#include <stddef.h>', '#include "dbslmm_b200.h"', 'int main(void) {']
    src += [f'  printf("{f} %zu\\n", offsetof(dbslmm_b200_fit_args, {f}));' for f in fields]
    src += [f'  printf("t.{f} %zu\\n", offsetof(dbslmm_b200_timing, {f}));' for f in tfields]
    src += ['  return 0;', '}']
    c = tmp_path / "off.c"
    c.write_text("\n".join(src))
    exe = tmp_path / "off"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(c), "-o", str(exe)], check=True)
    out = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip().split("\n"))
    for f in fields:
        assert int(out[f]) == getattr(_abi.FitArgs, f).offset, f
    for f in tfields:
        assert int(out["t." + f]) == getattr(_abi.Timing, f).offset, f
