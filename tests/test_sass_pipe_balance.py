"""Build-time guard for the pipe-balance ballast (csrc/dkg_mont.cuh: pipe_ballast): ptxas decides per
function whether register moves and carry adds go to the ALU pipe (MOV, IADD3.X) or to the multiplier
pipe (IMAD.MOV.U32, IMAD.X) -- the one pipe the exponentiation saturates.  A compiler change that
undoes the ballast's effect would silently cost ~5-15 % throughput; this test fails loudly instead.
Checked on the SASS of the headline kernels, modexp_nsq_kernel and modexp_nsq_multi_kernel at the shapes of 2048-bit-class keys, <13,5> and <14,5>,
inside their noinline Montgomery product (the target of their CALLs)."""
from __future__ import annotations

import collections
import os
import re
import shutil
import subprocess

import pytest


def _cuobjdump() -> str | None:
    """cuobjdump from PATH, else from the CUDA toolkit ($CUDA_HOME, /usr/local/cuda)."""
    for path in (shutil.which("cuobjdump"), *(os.path.join(h, "bin", "cuobjdump") for h in
                                              (os.environ.get("CUDA_HOME", ""), "/usr/local/cuda") if h)):
        if path and os.access(path, os.X_OK):
            return path
    return None


KERNELS = [("_ZN3dkg17modexp_nsq_kernelILi13ELi5ELb0EEEvNS_9NsqParamsE", 13),
           ("_ZN3dkg23modexp_nsq_multi_kernelILi13ELi5ELb0EEEvNS_14NsqMultiParamsE", 13),
           ("_ZN3dkg17modexp_nsq_kernelILi14ELi5ELb0EEEvNS_9NsqParamsE", 14),
           ("_ZN3dkg23modexp_nsq_multi_kernelILi14ELi5ELb0EEEvNS_14NsqMultiParamsE", 14)]


@pytest.mark.parametrize("KERNEL,K", KERNELS)
def test_hot_montgomery_product_keeps_the_multiplier_pipe_for_multiplies(KERNEL, K):
    from protocols.distributed_keygen_b200 import _native

    cuobjdump = _cuobjdump()
    if cuobjdump is None:
        pytest.skip("cuobjdump not found (PATH, $CUDA_HOME/bin, /usr/local/cuda/bin)")
    sass = subprocess.run([cuobjdump, "-sass", "-fun", KERNEL, _native.LIB_PATH], capture_output=True, text=True, check=True).stdout
    insts = [(int(m.group(1), 16), m.group(2)) for m in re.finditer(r"/\*([0-9a-f]{4,6})\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", sass)]
    assert len(insts) > 5000, "kernel not found in the library"
    targets = collections.Counter(int(t, 16) for t in re.findall(r"CALL\.REL\.NOINC\s+0x([0-9a-f]+)", sass))
    assert targets, "the Montgomery product is expected to be a noinline call"
    start = targets.most_common(1)[0][0]
    hot = [op for addr, op in insts if addr >= start]
    count = collections.Counter(op.split(".")[0] + ("." + op.split(".")[1] if op.startswith("IMAD.") else "") for op in hot)
    wide = sum(v for k, v in count.items() if k == "IMAD.WIDE")
    moves = count.get("IMAD.MOV", 0)
    carry_adds = count.get("IMAD.X", 0)
    assert wide >= K * K, f"expected the unrolled {K}x{K} block product, found {wide} IMAD.WIDE"
    assert moves == 0, f"{moves} IMAD.MOV on the multiplier pipe inside the hot function: the pipe ballast no longer works"
    assert carry_adds <= 16, f"{carry_adds} IMAD.X on the multiplier pipe inside the hot function (was 12)"
    # the ballast itself must still be there (never executed, it only tips ptxas's static balance)
    assert count.get("FFMA", 0) >= 1024
