"""The lanes physics kernel stages its walkers with every load of the prologue in flight at once.

Before the first substep each CTA copies its walkers' records, flags, step counters, positions, material ids, joint
torques and actions from global memory.  The kernel issues all of them as cp.async (SASS: LDGSTS) and waits once
(DEPBAR), so the prologue costs one memory round trip, not one per dependent load.  This test reads the SASS of the built
library: every global load before the wait is an LDGSTS, none comes after it, and no backward branch (a rolled loop that
would wait for each load in turn) sits between the kernel's entry and the wait.  It needs no GPU.
"""
import functools
import re

import pytest

from test_f32x2_sass_cpu import _sass_by_function

# cp.async instructions in the code at least: 3 for the record's rows (every layout has at least 3 pieces per lane) and
# 11 for one walker's other inputs
MIN_PIECES = 14
INSN = re.compile(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);")


@functools.lru_cache(maxsize=None)
def _sass(lib_path):
    return _sass_by_function(lib_path)


def _kernel(funcs, lanes, legs):
    name = [n for n in funcs if n.startswith(f"_ZN2wb2pl20physics_lanes_kernelILi{lanes}ELi{legs}ELb0")]
    assert len(name) == 1, f"physics_lanes_kernel<{lanes},{legs},0> not found in the library's SASS"
    code = []
    for line in funcs[name[0]]:
        m = INSN.match(line)
        if m:
            code.append((int(m.group(1), 16), m.group(2).strip()))
    return code


@pytest.mark.parametrize("lanes,legs", [(1, 1), (2, 2), (4, 2), (8, 2), (16, 2), (32, 2)])
def test_prologue_loads_all_in_flight_before_one_wait(wb, lanes, legs):
    code = _kernel(_sass(wb.lib()._name), lanes, legs)
    waits = [i for i, (_, op) in enumerate(code) if re.search(r"\bDEPBAR\b", op)]
    assert waits, "no cp.async wait (DEPBAR) in the kernel"
    first_wait = waits[0]
    before = [op for _, op in code[:first_wait]]
    assert sum(" LDGSTS" in f" {op}" for op in before) >= MIN_PIECES
    plain = [op for op in before if re.search(r"\bLDG\b|\bLDG\.", op)]
    assert not plain, f"global loads before the wait that are not cp.async: {plain}"
    late = [op for _, op in code[first_wait:] if "LDGSTS" in op]
    assert not late, f"cp.async after the first wait: {late}"
    for addr, op in code[:first_wait]:
        m = re.search(r"\bBRA(?:\.\S+)?\s+(?:!?U?P\w+,\s*)?(0x[0-9a-f]+)", op)
        assert not (m and int(m.group(1), 16) <= addr), f"backward branch before the wait at {addr:#x}: {op}"
