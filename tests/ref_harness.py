"""
Test harness that runs the REFERENCE's own ``DistributedPaillier`` / ``PaillierSharedKey`` code in
one process: where the unmodified reference is importable (``baseline/_ref``, the git-ignored pip
``--target`` install recorded in DESIGN.md, or the ``src`` directory of a checkout of the reference
named by ``DKG_REFERENCE_SRC``), its un-vendored third-party imports are satisfied by the
data-holder shims in ``tests/golden/ref_shims`` and the parties talk through the in-process
``FakePool`` below instead of ``tno.mpc.communication``'s HTTP pool (API used by the reference:
``async_broadcast``, ``recv_all``; ``distributed_keygen.py:357-370, 476-496``).  The repository
does not contain the reference: without a copy, the tests that use this harness skip.  Test
infrastructure only.
"""
from __future__ import annotations

import asyncio
import base64
import importlib
import os
import sys
from typing import Any

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIMS = os.path.join(ROOT, "tests", "golden", "ref_shims")
CANDIDATES = [os.path.join(ROOT, "baseline", "_ref"), os.environ.get("DKG_REFERENCE_SRC")]


def import_reference() -> Any:
    """The reference package, or ``None`` when no copy of it is reachable from here."""
    for path in CANDIDATES:
        if path and os.path.isdir(os.path.join(path, "tno", "mpc", "protocols", "distributed_keygen")):
            for extra in (SHIMS, path):
                if extra not in sys.path:
                    sys.path.insert(0, extra)
            return importlib.import_module("tno.mpc.protocols.distributed_keygen")
    return None


class FakeHub:
    """Shared mailbox of the in-process parties."""

    def __init__(self, names: list[str]) -> None:
        self.names = names
        self.box: dict[tuple[str, str], dict[str, Any]] = {}
        self.cond: asyncio.Condition | None = None
        self.sent = 0


class FakePool:
    """One party's view: ``pool_handlers`` are the OTHER parties' names."""

    def __init__(self, hub: FakeHub, me: str) -> None:
        self.hub, self.me = hub, me
        self.pool_handlers = {n: object() for n in hub.names if n != me}

    def async_broadcast(self, message: Any, msg_id: str, handler_names: list[str] | None = None) -> None:
        for name in (self.pool_handlers if handler_names is None else handler_names):
            self.hub.box.setdefault((name, msg_id), {})[self.me] = message
            self.hub.sent += 1

    async def recv_all(self, msg_id: str) -> tuple[tuple[str, Any], ...]:
        while True:
            got = self.hub.box.get((self.me, msg_id), {})
            if len(got) == len(self.pool_handlers):
                del self.hub.box[(self.me, msg_id)]
                return tuple(got.items())
            await asyncio.sleep(0)


def make_schemes(ref: Any, key_entries: list[dict], t: int, precision: int = 8, session_id: int = 77) -> dict[int, Any]:
    """One reference ``DistributedPaillier`` per party, built on the reference's own stored-key
    fixtures (``tests/golden/fixture_vectors.json`` holds the blobs) -- the in-process equivalent
    of the ``distributed_schemes`` fixture of the reference's tests (``test/conftest.py:94-134``)."""
    from tno.mpc.encryption_schemes.paillier import PaillierPublicKey
    from tno.mpc.encryption_schemes.shamir import IntegerShares, ShamirSecretSharingIntegers

    from protocols.distributed_keygen_b200.keyio import load_private_key_from_bytes

    stored = [load_private_key_from_bytes(base64.b64decode(e["blob_b64"])) for e in key_entries]
    names = {s.secret_key.player_id: f"local{s.secret_key.player_id}" for s in stored}
    hub = FakeHub(list(names.values()))
    schemes = {}
    for s, e in zip(stored, key_entries):
        k = s.secret_key
        scheme = ShamirSecretSharingIntegers(e["kappa"], k.n, len(stored), t)
        ref_key = ref.PaillierSharedKey(
            n=k.n, t=k.t, player_id=k.player_id,
            share=IntegerShares(scheme, dict(k.share.shares), k.share.degree, k.share.scaling), theta=k.theta,
        )
        party_indices = {("self" if pid == k.player_id else nm): pid for pid, nm in names.items()}
        schemes[k.player_id] = ref.DistributedPaillier(
            PaillierPublicKey(k.n, k.n + 1), ref_key, precision, FakePool(hub, names[k.player_id]),
            k.player_id, party_indices, session_id, False, t,
        )
        k.close()
    return schemes


def ciphertext(scheme: Any, raw: int) -> Any:
    from tno.mpc.encryption_schemes.paillier import PaillierCiphertext

    return PaillierCiphertext(raw, scheme)


def encode(m: float, n: int, precision: int = 8) -> int:
    """Fixed-point encoding of the third-party scheme (SURVEY appendix A): m * 10^precision mod N."""
    return round(m * 10**precision) % n


def decode(v: int, n: int, precision: int = 8) -> float:
    signed = v if v <= n // 2 else v - n
    return signed / 10**precision


def run(coro_list: list[Any]) -> list[Any]:
    async def go() -> list[Any]:
        return list(await asyncio.gather(*coro_list))

    return asyncio.run(go())
