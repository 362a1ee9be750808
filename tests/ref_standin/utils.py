"""``Batched`` / ``AdditiveVariable`` of the reference's utils, as data holders (see the package
docstring): the patched biprime v calculation returns its values in them."""
from typing import Any


class AdditiveVariable:
    def __init__(self, label: str, modulus: int) -> None:
        self.label = label
        self.modulus = modulus


class Batched:
    def __init__(self, variable: Any, batch_size: int) -> None:
        self.variable = variable
        self.batch_size = batch_size
        self.shares: dict[int, list[int]] = {}

    def set_share(self, index: int, values: list[int]) -> None:
        self.shares[index] = list(values)

    def get_share(self, index: int) -> list[int]:
        return self.shares[index]
