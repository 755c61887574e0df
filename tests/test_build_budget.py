"""Resource budget of the decode-program kernel, checked from ptxas on the CPU box (nvcc cross-compiles sm_100a here):
one CTA of 320 threads per SM must fit the register file (65536 / 320 = 204 registers per thread) without spilling -
a spill in the tile loop, or a register count that drops the launch to zero resident CTAs, would only show up on the
GPU otherwise."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("nvcc") is None, reason="needs nvcc")
def test_program_kernels_register_and_spill_budget(tmp_path):
    src = os.path.join(ROOT, "autoawq_b200", "csrc", "program.cu")
    out = subprocess.run(
        ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xptxas", "-v", "-c", src,
         "-o", str(tmp_path / "program.o")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-2000:]
    log = out.stderr + out.stdout
    entries = re.findall(r"Compiling entry function '(\S*program_kernel\S*)'[^\n]*\n[^\n]*\n\s*(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores, (\d+) bytes spill loads\n[^\n]*Used (\d+) registers", log)
    assert len(entries) == 2, log[-1500:]          # program_kernel<2>, stream_program_kernel<8 warps>
    assert sum("stream_program_kernel" in e[0] for e in entries) == 1
    for name, stack, st, ld, regs in entries:
        if "stream_program_kernel" in name:
            # one resident CTA of 32 + 32 NW threads; a few spilled words in the staging phase (off the unit loop) are
            # tolerated, a spilling unit loop is not: keep the total small
            nw = int(re.search(r"kernelILi(\d+)E", name).group(1))
            assert int(regs) * (32 + 32 * nw) <= 65536, f"{name}: {regs} registers x {32 + 32 * nw} threads"
            assert int(st) <= 128 and int(ld) <= 256, f"{name}: spills {st} / {ld} bytes"
        else:
            assert int(st) == 0 and int(ld) == 0 and int(stack) == 0, f"{name}: spills"
            assert int(regs) <= 204, f"{name}: {regs} registers x 320 threads exceed the register file"


@pytest.mark.skipif(shutil.which("nvcc") is None, reason="needs nvcc")
def test_tcgen05_kernels_register_budget(tmp_path):
    """One CTA per SM: gemm_tc_kernel runs 448 threads, gemm_tcq_kernel 768 - registers x threads must fit the 64 K register file and nothing may spill (the small-M
    kernel's producer loop is issue-bound: a spill there is a measurable loss, and 3 Q-TMA warps = 800 threads capped the
    allocation at 72 registers and DID spill, which is why there is one)."""
    src = os.path.join(ROOT, "autoawq_b200", "csrc", "gemm_tc.cu")
    out = subprocess.run(
        ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xptxas", "-v", "-c", src,
         "-o", str(tmp_path / "gemm_tc.o")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr[-2000:]
    log = out.stderr + out.stdout
    entries = re.findall(r"Compiling entry function '(\S*gemm_tcq?_kernel\S*)'[^\n]*\n[^\n]*\n\s*(\d+) bytes stack frame, "
                         r"(\d+) bytes spill stores, (\d+) bytes spill loads\n[^\n]*Used (\d+) registers", log)
    tcq = [e for e in entries if "gemm_tcq_kernel" in e[0]]
    tc = [e for e in entries if "gemm_tcq_kernel" not in e[0]]
    assert len(tcq) == 4 and len(tc) == 16, (len(tcq), len(tc))     # BT in {16, 32, 64, 128}; 4 token tiles x 4 layouts
    for name, stack, st, ld, regs in tcq:
        assert int(st) == 0 and int(ld) == 0 and int(stack) == 0, f"{name}: spills"
        assert int(regs) * 768 <= 65536, f"{name}: {regs} registers x 768 threads"
    for name, stack, st, ld, regs in tc:
        assert int(st) == 0 and int(ld) == 0, f"{name}: spills"
        assert int(regs) * 448 <= 65536, f"{name}: {regs} registers x 448 threads"
