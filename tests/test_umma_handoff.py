"""tests/cpp/umma_probe3.cu: the A-operand hand-off of DecoderKernelDU's residual units (an A operand in tensor memory read
by MMAs, tcgen05.commit to an mbarrier, the columns overwritten with the next k-half after the wait, further MMAs into the same
accumulator).  On the hardware it pins the write-after-read ordering; on the emulator, which executes MMAs at issue, the
column arithmetic."""
import os
import subprocess

import pytest

from conftest import EMU_DIR, ROOT

PROBE = os.path.join(ROOT, "tests", "cpp", "umma_probe3.cu")


def _check(out):
    assert out.returncode == 0 and out.stdout.count("MATCH") == 1 and "MISMATCH" not in out.stdout, out.stdout + out.stderr


def test_emu_umma_handoff_probe(tmp_path):
    exe = str(tmp_path / "umma_probe3")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-DLYRA_EMU", "-x", "c++", "-I" + EMU_DIR, "-I" + os.path.join(ROOT, "lyra_b200", "csrc"),
                           "-Wno-unknown-pragmas", PROBE, os.path.join(EMU_DIR, "cuda_emu.cc"), "-o", exe])
    _check(subprocess.run([exe], capture_output=True, text=True, timeout=300))


@pytest.mark.gpu
def test_umma_handoff_probe_on_hardware(tmp_path):
    import __graft_entry__ as g
    exe = str(tmp_path / "umma_probe3")
    subprocess.check_call([g.NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I" + os.path.join(ROOT, "lyra_b200", "csrc"),
                           "-o", exe, PROBE])
    out = subprocess.run(["timeout", "60", exe], capture_output=True, text=True, timeout=120)
    print(out.stdout.strip())
    _check(out)
