"""``DistributedPaillier`` of the reference, names and constructor only (see the package docstring)."""
from typing import Any

from tno.mpc.encryption_schemes.templates import EncodedPlaintext  # noqa: F401  (read by the patch)


class DistributedPaillier:
    def __init__(self, public_key: Any, secret_key: Any, precision: int, pool: Any, index: int,
                 party_indices: dict, session_id: int, distributed: bool, corruption_threshold: int) -> None:
        self.public_key = public_key
        self.secret_key = secret_key
        self.precision = precision
        self.pool = pool
        self.index = index
        self.party_indices = party_indices
        self.session_id = session_id
        self.distributed = distributed
        self.corruption_threshold = corruption_threshold

    async def _decrypt_sequence_raw(self, ciphertext_sequence: Any, receivers: Any = None) -> Any:
        raise NotImplementedError("stand-in: only the patched method computes")

    @classmethod
    def __biprime_test_v_calculation(cls, g_values: Any, index: int, modulus: int, p_i: int, q_i: int,
                                     correct_param_biprime: int) -> Any:
        raise NotImplementedError("stand-in: only the patched method computes")
