"""CPU check of the kernel instance matrix (tests/kernel_matrix.py): the cases of the table, taken together, make every kernel instance
compiled into libb2align.so serve a pair -- no more, no fewer.  The instance list comes from the library itself (`cuobjdump -symbols`,
demangled with `cu++filt`), so a new template instance without a case, or a case naming an instance that no longer exists, fails here
with the instances' names."""
import os
import re
import shutil
import subprocess

import pytest

import kernel_matrix as km
from __graft_entry__ import load_package

pkg = load_package()
EXCLUDED = {"microbench_kernel"}                  # device-rate microbenchmarks (b2a_microbench_int16x2), no alignment work


def cuda_tool(name):
    for d in (os.environ.get("CUDA_HOME"), os.environ.get("CUDA_PATH"), "/usr/local/cuda"):
        if d and os.path.exists(os.path.join(d, "bin", name)):
            return os.path.join(d, "bin", name)
    path = shutil.which(name)
    assert path, f"{name} (CUDA toolkit) not found"
    return path


def parse_entry(sym):
    """'void b2a::short16_fill_kernel<(int)16, (int)8, (bool)0, (bool)1, (bool)0>(b2a::FillArgs)' -> ('short16_fill_kernel', (16, 8, 0, 1, 0))"""
    m = re.match(r"(?:void )?(?:<unnamed>::|\(anonymous namespace\)::|b2a::)*(\w+)(?:<([^>]*)>)?\(", sym)
    assert m, sym
    args = tuple(int(x) for x in re.findall(r"\((?:int|bool)\)(-?\d+)", m.group(2) or ""))
    return m.group(1), args


def library_instances():
    raw = subprocess.run([cuda_tool("cuobjdump"), "-symbols", pkg.LIB_PATH], capture_output=True, text=True, check=True).stdout
    dem = subprocess.run([cuda_tool("cu++filt")], input=raw, capture_output=True, text=True, check=True).stdout
    out = set()
    for line in dem.splitlines():
        if "STO_ENTRY" in line:
            out.add(parse_entry(line.split("STO_ENTRY", 1)[1].strip()))
    return out


def fmt(inst):
    name, args = inst
    return f"{name}<{', '.join(map(str, args))}>" if args else name


def test_parse_entry():
    assert parse_entry("void b2a::wide32_fill_kernel<(int)2, (bool)1, (bool)0, (bool)1, (bool)1, (bool)0>(b2a::WideArgs)") == \
        ("wide32_fill_kernel", (2, 1, 0, 1, 1, 0))
    assert parse_entry("<unnamed>::dirty_kernel(const unsigned char *, const unsigned long *)") == ("dirty_kernel", ())
    assert parse_entry("b2a::wide32_first_best_row_kernel(const unsigned int *, unsigned int, b2a::CkptWalk *)") == \
        ("wide32_first_best_row_kernel", ())


def test_case_table_reaches_every_kernel_instance_of_the_library():
    if not os.path.exists(pkg.LIB_PATH):
        pytest.skip("libb2align.so not built")
    have = {i for i in library_instances() if i[0] not in EXCLUDED}
    assert len(have) > 250
    covered = set()
    for case in km.all_cases():
        covered |= km.instances(case)
    missing, unknown = sorted(have - covered), sorted(covered - have)
    msg = []
    if missing:
        msg.append("kernel instances without a case in tests/kernel_matrix.py: " + ", ".join(map(fmt, missing)))
    if unknown:
        msg.append("instances named by a case that the library does not have: " + ", ".join(map(fmt, unknown)))
    assert not msg, "; ".join(msg)


def test_case_table_shapes():
    """the edges the table promises: every rows-per-lane class at both ends in both short16 symbol variants, pair-pairs of one shape,
    mixed-shape pair-pairs and singletons in every class, and each plan-boundary pair on the side of the boundary it is meant for"""
    for case in km.short16_cases():
        pps, wide = km.pair_pairs(case)
        assert set(pps) == set(km.R_CLASSES), case.name
        for R, lst in pps.items():
            shapes = [(len(case.pairs[a][0]), len(case.pairs[a][1])) == (len(case.pairs[b][0]), len(case.pairs[b][1])) for a, b in lst]
            assert any(a != b and same for (a, b), same in zip(lst, shapes)), (case.name, R)        # same-shape pair-pair
            assert any(a != b and not same for (a, b), same in zip(lst, shapes)), (case.name, R)    # mixed-shape pair-pair
            assert any(a == b for a, b in lst), (case.name, R)                                       # singleton
        fills = {i[1][:4] for i in km.instances(case) if i[0] == "short16_fill_kernel"}
        assert {(R, a8) for R, _, _, a8 in fills} == {(R, a8) for R in km.R_CLASSES for a8 in (0, 1)}, case.name
        _, path = km.route(case)
        assert path[-1] == path[-2] == 2 and path.count(2) == 2, case.name                     # only the 8-symbol pair-pair leaves short16
    for case in km.boundary_cases():
        _, path = km.route(case)
        assert path == [1, 1, 2, 2] * len(km.R_CLASSES), case.name
