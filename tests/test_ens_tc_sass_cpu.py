"""CPU: the machine code of the two tcgen05 kernels the rollout spends its time in (K1, the 512-wide swish dynamics
ensemble as cluster pairs, and the merged policy pass, grouped with run-time activations) keeps its shared-memory
operands in the shared state space (no generic LD / ST anywhere, so none inside a drain either) and its registers out
of local memory.

A shared pointer rebuilt from an integer turns every bias and scaler read into a generic, long-scoreboard LD.E, and a
spilled unit counter turns every unit boundary into LDL / STL; both sat on the epilogue's drain chain before.  Reads
build/ens_tc.o (left by build.sh); skips when the object or cuobjdump is absent."""
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "build", "ens_tc.o")

# ens_mlp3_tc_kernel<HD, FMT, ACT, G, NMID, CL, WO>: FMT 0 = fp16, 1 = bf16; ACT 1 = swish, 0 = per-member
KERNELS = {
    "k1_fp16": "ens_mlp3_tc_kernelILi512ELi0ELi1ELi1ELi0ELi2ELb0E",
    "k1_bf16": "ens_mlp3_tc_kernelILi512ELi1ELi1ELi1ELi0ELi2ELb0E",
    "policy_fp16": "ens_mlp3_tc_kernelILi512ELi0ELi0ELi4ELi0ELi1ELb0E",
    "policy_bf16": "ens_mlp3_tc_kernelILi512ELi1ELi0ELi4ELi0ELi1ELb0E",
}


def _cuobjdump():
    for c in (shutil.which("cuobjdump"), os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")):
        if c and os.access(c, os.X_OK):
            return c
    return None


@pytest.fixture(scope="module")
def sass():
    tool = _cuobjdump()
    if not os.path.exists(OBJ) or tool is None:
        pytest.skip("needs build/ens_tc.o and cuobjdump")
    text = subprocess.run([tool, "-sass", OBJ], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in text.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Za-z0-9_.]*)", line)
        if m and cur is not None:
            cur.append(m.group(1))
    return funcs


def _ops(sass, key):
    names = [n for n in sass if KERNELS[key] in n]
    assert len(names) == 1, (key, names)
    ops = sass[names[0]]
    assert "UTCHMMA" in ops and "LDTM.x16" in ops and "STTM.x16" in ops, key
    return ops


@pytest.mark.parametrize("key", sorted(KERNELS))
def test_no_local_memory(sass, key):
    local = [o for o in _ops(sass, key) if o.split(".")[0] in ("LDL", "STL")]
    assert not local, (key, local)


@pytest.mark.parametrize("key", sorted(KERNELS))
def test_drain_reads_shared_memory_as_shared(sass, key):
    ops = _ops(sass, key)
    generic = [o for o in ops if o.split(".")[0] in ("LD", "ST")]
    assert not generic, (key, generic)
    assert "LDS.128" in ops, key                  # the drain's biases: broadcast shared-memory loads
