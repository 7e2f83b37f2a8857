"""The physics kernels use the paired fp32 instructions of sm_100 and contain no fused multiply-add of a pair.

The physics translation units are compiled with -fmad=false: every product and sum is rounded on its own (bit-exact
contract, DESIGN §4.1).  ptxas nevertheless contracts an add.rn.f32x2 that consumes a mul.rn.f32x2 into one FFMA2, which
rounds once.  physics_math.cuh keeps paired products away from paired sums; this test reads the SASS of the built library
and fails if an FFMA2 appears in a physics kernel.  It needs no GPU: cuobjdump reads the sm_100a code from the library.
"""
import os
import re
import shutil
import subprocess

# wb::pl (lanes kernels), wb::pc (compacting kernel), wb::sc (scene and terrain kernels)
PHYSICS = re.compile(r"^_ZN2wb2(pl|pc|sc)")


def _cuobjdump():
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand and os.path.exists(cand):
            return cand
    nvcc = shutil.which("nvcc")
    assert nvcc, "cuobjdump not found (CUDA toolkit)"
    return os.path.join(os.path.dirname(nvcc), "cuobjdump")


def _sass_by_function(lib_path):
    out = subprocess.run([_cuobjdump(), "-sass", lib_path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur is not None and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):
            funcs[cur].append(line)
    return funcs


def test_physics_kernels_pair_fp32_without_contraction(wb):
    funcs = _sass_by_function(wb.lib()._name)
    physics = {name: code for name, code in funcs.items() if PHYSICS.match(name)}
    assert any("physics_lanes_kernel" in n for n in physics), "no physics kernel found in the library's SASS"
    fused = {name: sum(" FFMA2 " in l for l in code) for name, code in physics.items()}
    fused = {name: n for name, n in fused.items() if n}
    assert not fused, f"FFMA2 (a contracted paired multiply-add) in physics kernels: {fused}"
    # the headline layout (8 lanes per walker, 2 walkers per warp) issues its vector sums and products as pairs
    k82 = [code for name, code in physics.items() if name.startswith("_ZN2wb2pl20physics_lanes_kernelILi8ELi2ELb0")]
    assert len(k82) == 1
    assert sum(" FADD2 " in l for l in k82[0]) > 0 and sum(" FMUL2 " in l for l in k82[0]) > 0
