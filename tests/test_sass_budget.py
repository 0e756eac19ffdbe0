"""Static evidence from the built library, checked on the CPU box: the instructions that prove which hardware path a kernel uses
(the SASS mnemonics of B200_PROFILING.md) and the register / spill budget the measured occupancy of the hot kernels rests on
(`ptxas -v` logs of the in-tree build).  A kernel edit that silently falls off the tensor cores, loses the cp.async staging or
blows the register budget (28 resident one-warp blocks per SM need <= 72 registers) fails here before it costs a GPU minute."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "seganygaussians_b200", "lib", "obj")

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None or not os.path.isdir(OBJ), reason="needs cuobjdump and the in-tree build")


def _sass(obj):
    return subprocess.run(["cuobjdump", "-sass", os.path.join(OBJ, obj)], capture_output=True, text=True, check=True).stdout


def _functions(sass):
    out, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur is not None:
            out[cur].append(line)
    return {k: "\n".join(v) for k, v in out.items()}


def _ptxas(log):
    """entry name -> (registers, spill store bytes, spill load bytes)"""
    txt = open(os.path.join(OBJ, log)).read()
    res = {}
    for m in re.finditer(r"Compiling entry function '(\S+)' for 'sm_100a'.*?(\d+) bytes spill stores, (\d+) bytes spill loads.*?Used (\d+) registers", txt, re.S):
        res[m.group(1)] = (int(m.group(4)), int(m.group(2)), int(m.group(3)))
    return res


def test_every_object_carries_sm100a_code_only():
    for obj in sorted(f for f in os.listdir(OBJ) if f.endswith(".o")):
        out = subprocess.run(["cuobjdump", "-lelf", os.path.join(OBJ, obj)], capture_output=True, text=True).stdout
        archs = set(re.findall(r"sm_(\d+a?)", out))
        assert archs <= {"100a"}, (obj, archs)


def test_tensor_core_and_copy_engine_mnemonics():
    f = _functions(_sass("render_forward_warp.o"))
    k = next(v for n, v in f.items() if "render_forward_warp_kernelILi8ELb1E" in n)
    assert k.count("HMMA.1688.F32.TF32") >= 24                       # 2 m-tiles x 4 n-tiles x 3 (3xTF32) per group of 8 candidates
    f = _functions(_sass("render_backward_warp.o"))
    k = next(v for n, v in f.items() if "render_backward_warp_kernelILi8ELb1ELb0ELb1" in n)
    assert k.count("HMMA.1688.F32.TF32") >= 56 and "REDG.E.ADD.F32" in k   # dot products + colour product + moments; fire-and-forget adds
    tc = _sass("render_forward_tc.o")
    assert "UTCHMMA" in tc and "LDTM" in tc                             # tcgen05.mma with TMEM accumulators, tcgen05.ld epilogue
    f = _functions(_sass("render_forward.o"))
    plain = [v for n, v in f.items() if "render_forward_kernelI" in n]
    assert plain and all("LDGSTS" in v and "UBLKCP" not in v for v in plain)
    assert "LDGMC.E.ADD.F32x4" in _sass("multimem_allreduce.o")         # multimem.ld_reduce: the in-switch reduction


def test_register_budget_of_the_hot_kernels():
    bw = _ptxas("render_backward_warp.ptxas.log")
    fw = _ptxas("render_forward_warp.ptxas.log")
    regs, st, ld = next(v for n, v in bw.items() if "render_backward_warp_kernelILi8ELb1ELb0ELb1" in n)
    assert regs <= 72 and st <= 32 and ld <= 32, (regs, st, ld)        # 28 one-warp blocks per SM; the measured build spills 28 / 32 B
    regs, st, ld = next(v for n, v in fw.items() if "render_forward_warp_kernelILi8ELb1E" in n)
    assert regs <= 72 and st <= 32 and ld <= 32, (regs, st, ld)
    for log in ("preprocess.ptxas.log", "binning.ptxas.log", "geom_backward.ptxas.log", "tile_sort.ptxas.log", "smooth.ptxas.log"):
        for name, (regs, st, ld) in _ptxas(log).items():
            assert st == 0 and ld == 0, (log, name, st, ld)             # the streaming kernels must not spill at all
