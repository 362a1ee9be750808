"""``PaillierSharedKey`` of the reference, names only (see the package docstring)."""
from typing import Any

from tno.mpc.encryption_schemes.paillier import PaillierCiphertext  # noqa: F401  (read by the patch)


class PaillierSharedKey:
    def __init__(self, n: int, t: int, player_id: int, share: Any, theta: int) -> None:
        self.n = n
        self.t = t
        self.player_id = player_id
        self.share = share
        self.theta = theta
        self.n_square = n * n

    def partial_decrypt(self, ciphertext: Any) -> int:
        raise NotImplementedError("stand-in: only the patched method computes")

    def decrypt(self, partial_dict: Any) -> int:
        raise NotImplementedError("stand-in: only the patched method computes")
