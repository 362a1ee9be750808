"""
Stand-in for the interface of the reference package ``tno.mpc.protocols.distributed_keygen`` that
``protocols.distributed_keygen_b200.patch`` binds to: the modules ``distributed_keygen``,
``paillier_shared_key`` and ``utils`` with the class and attribute names the patch rebinds or reads,
and the constructor arguments ``tests/ref_harness.make_schemes`` passes.  It is NOT the reference
and holds no arithmetic: the methods the patch replaces raise here, so every value a test sees comes
from the patched (engine) code.  Tests compare those values with the ones recorded from the
reference's own classes (``tests/golden/*.json``).  Like the reference, it imports its third-party
packages, which the shims in ``tests/golden/ref_shims`` provide.
"""
import os
import sys

_SHIMS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden", "ref_shims")
if _SHIMS not in sys.path:
    sys.path.insert(0, _SHIMS)

from .distributed_keygen import DistributedPaillier  # noqa: E402,F401
from .paillier_shared_key import PaillierSharedKey  # noqa: E402,F401
