"""Guards on what ptxas made of the hot kernels (uav-autonomous-control_b200/lib/build.log, written by build.py): the persistent
rollout kernels must not keep state in local memory.  (Round 2: one extra inlined call site of the flying code made ptxas copy the
kernel parameter block to the stack in six of eight instantiations -- 1280-byte frames, BASELINE configs[3] 108 -> 191 ms -- without
any test noticing.)  Also: what the built library itself contains."""
from __future__ import annotations

import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LOG = os.path.join(ROOT, "uav-autonomous-control_b200", "lib", "build.log")
LIB = os.path.join(ROOT, "uav-autonomous-control_b200", "lib", "libuavb.so")


def _kernels():
    text = open(LOG).read()
    pat = re.compile(r"Function properties for (\S+)\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\s+"
                     r"ptxas info\s+: Used (\d+) registers")
    return [(m.group(1), int(m.group(2)), int(m.group(3)), int(m.group(5))) for m in pat.finditer(text)]


@pytest.mark.skipif(not os.path.exists(LOG), reason="library not built in this tree")
def test_rollout_kernels_keep_their_state_in_registers():
    ks = [k for k in _kernels() if "rollout_sliced" in k[0]]
    assert len(ks) >= 24                                          # metrics-only, per-thread log, tensor-store log, trajectory list
    for name, stack, spill, regs in ks:
        allowed = 64 if "scalar" in name else 0                 # the 128-register one-drone-per-thread kernel spills a few words
        assert stack <= (96 if "scalar" in name else 64) and spill <= allowed, f"{name}: {stack} B stack frame, {spill} B spills at {regs} registers"
    headline = [k for k in ks if "rollout_sliced_kernelILb1ELb1ELb0ELb1" in k[0]]
    assert headline and headline[0][1] == 0 and headline[0][3] <= 255


@pytest.mark.skipif(not os.path.exists(LOG), reason="library not built in this tree")
def test_streaming_solver_fits_four_ctas_per_sm():
    ks = [k for k in _kernels() if "minsnap_solve_stream_kernelILi4" in k[0]]
    assert ks and ks[0][3] <= 255 and ks[0][2] <= 64             # 4 CTAs x 64 threads x 255 registers; a handful of spilled bytes at most


@pytest.mark.skipif(not os.path.exists(LIB), reason="library not built in this tree")
def test_library_reads_no_slicing_overrides_from_the_environment():
    """How a rollout launch is sliced is fixed in the code: no variable in the user's environment changes it."""
    with open(LIB, "rb") as f:
        data = f.read()
    for name in (b"UAVB_ROLLOUT_CHUNKS", b"UAVB_SLICE_MIN", b"UAVB_SLICE_PART"):
        assert name not in data, name.decode()
