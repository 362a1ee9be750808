"""CPU-only checks of the host side: the C-ABI library loads and exports every symbol the header
declares, compute entry points fail loudly without a GPU (no CPU fallback), limb packing, the
per-key exponent against the oracle, the Jacobi filter, index sharding."""
from __future__ import annotations

import base64
import ctypes
import os
import random
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from protocols.distributed_keygen_b200 import _native

    header = open(os.path.join(ROOT, "include", "dkg_b200.h")).read()
    declared = set(re.findall(r"\b(dkg_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_native.EXPORTS), declared ^ set(_native.EXPORTS)
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _native.lib.dkg_version() >= 100


_NO_DEVICE_CHECK = """
import sys
sys.path.insert(0, sys.argv[1])
import pytest
import protocols.distributed_keygen_b200 as eng
from protocols.distributed_keygen_b200 import _native

assert _native.device_count() == 0
with pytest.raises(_native.DkgError) as err:
    eng.ModexpContext(35, 3)
assert err.value.code == _native.DKG_ERR_CUDA
with pytest.raises(_native.DkgError):
    eng.modexp_grouped([35], [3], [[2]])
"""


def test_no_cpu_fallback_without_device():
    """Runs in a child process with every device hidden (CUDA_VISIBLE_DEVICES empty), so that the
    no-device path is also checked on machines that have a GPU."""
    res = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHECK, ROOT], capture_output=True, text=True,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert res.returncode == 0, res.stderr


def test_argument_validation():
    import protocols.distributed_keygen_b200 as eng

    with pytest.raises(ValueError):
        eng.ModexpContext(36, 3)  # even modulus
    with pytest.raises(ValueError):
        eng.modexp_grouped([36], [3], [[2]])


def test_limb_packing_roundtrip():
    from protocols.distributed_keygen_b200.limbs import (
        int_to_limbs, ints_to_limbs, limbs_for_bits, limbs_to_int, limbs_to_ints,
    )

    rng = random.Random(1)
    vals = [0, 1, 2**32 - 1, 2**32, rng.getrandbits(4100)]
    arr = ints_to_limbs(vals, 129)
    assert arr.shape == (5, 129) and limbs_to_ints(arr) == vals
    assert limbs_to_int(int_to_limbs(vals[-1], 129)) == vals[-1]
    assert limbs_for_bits(4096) == 128 and limbs_for_bits(4097) == 129 and limbs_for_bits(0) == 1
    # little-endian limb order == int.to_bytes(..., "little")
    assert arr[3, 0] == 0 and arr[3, 1] == 1


def test_partial_decrypt_exponent_matches_oracle(fixture_vectors, dealer_vectors):
    from oracle import keys as okeys
    from protocols.distributed_keygen_b200 import IntegerShares, PaillierSharedKey

    oracle_keys = []
    for entry in fixture_vectors["sets"]:
        oracle_keys += [okeys.key_from_blob(base64.b64decode(k["blob_b64"])) for k in entry["keys"]]
    for item in dealer_vectors["keys"].values():
        oracle_keys += list(okeys.dealer_key_from_json(item["key"]).keys.values())
    assert len(oracle_keys) >= 24
    for k in oracle_keys:
        share = IntegerShares(dict(k.share.shares), k.share.degree, k.share.scaling, k.share.number_of_parties)
        key = PaillierSharedKey(k.n, k.t, k.player_id, share, k.theta)
        assert key.partial_decrypt_exponent() == k.partial_decrypt_exponent()
        assert key.theta_inv == k.theta_inv and key.n_square == k.n_square


def test_jacobi_and_biprime_host_logic(biprime_vectors):
    import sympy

    from oracle import paillier_oracle as po
    from protocols.distributed_keygen_b200 import distributed_keygen as dkg

    rng = random.Random(3)
    for _ in range(300):   # the oracle's Jacobi symbol (the product computes it on the GPU only)
        n = rng.getrandbits(rng.choice([8, 40, 200])) | 1
        a = rng.getrandbits(210)
        assert sympy.jacobi_symbol(a, n) == po.jacobi(a, n)
    assert not hasattr(dkg, "jacobi_symbol") and not hasattr(dkg, "_select_g"), "no host-side filter in the product"
    for case in biprime_vectors["cases"]:
        n = int(case["n"], 16)
        g_values = [int(g, 16) for g in case["g_values"]]
        correct = case["correct_param_biprime"]
        for i in range(1, case["parties"] + 1):
            p_i, q_i = int(case["p_shares"][i - 1], 16), int(case["q_shares"][i - 1], 16)
            assert dkg.biprime_exponent(i, n, p_i, q_i) == po.biprime_exponent(i, n, p_i, q_i)
        v_by_party = {int(p): [int(v, 16) for v in vs] for p, vs in case["v"].items()}
        if all(len(v) >= correct for v in v_by_party.values()):
            assert dkg.biprime_test_with_v_i(v_by_party, n, correct) == case["verdict"]


def test_shard_bounds():
    from protocols.distributed_keygen_b200.sharding import all_shards, shard_bounds

    for count in [0, 1, 7, 8, 1000, 10**7 + 3]:
        for world in [1, 2, 3, 8]:
            shards = all_shards(count, world)
            assert shards[0][0] == 0 and shards[-1][1] == count
            assert all(a[1] == b[0] for a, b in zip(shards, shards[1:]))
            sizes = [hi - lo for lo, hi in shards]
            assert max(sizes) - min(sizes) <= 1
    # group-granular: 40 bases of a candidate stay together
    shards = all_shards(40 * 13, 8, granule=40)
    assert all(lo % 40 == 0 and hi % 40 == 0 for lo, hi in shards) and shards[-1][1] == 520
    with pytest.raises(ValueError):
        shard_bounds(10, 2, 2)


def test_key_blob_reader_on_reference_fixtures(fixture_vectors):
    """The 24 stored keys of the reference's test suite through the product's own reader."""
    from oracle import keys as okeys
    from protocols.distributed_keygen_b200.keyio import load_private_key_from_bytes

    seen = 0
    for entry in fixture_vectors["sets"]:
        for k in entry["keys"]:
            blob = base64.b64decode(k["blob_b64"])
            stored = load_private_key_from_bytes(blob)
            want = okeys.key_from_blob(blob)
            key = stored.secret_key
            assert (key.n, key.t, key.player_id, key.theta) == (want.n, want.t, want.player_id, want.theta)
            assert key.share.shares == want.share.shares and key.share.degree == want.share.degree
            assert stored.g == stored.n + 1 and stored.corruption_threshold == entry["t"]
            assert stored.index == key.player_id and stored.precision == 8
            assert key.partial_decrypt_exponent() == want.partial_decrypt_exponent()
            seen += 1
    assert seen == 24


def test_oracle_is_test_infrastructure_only():
    """Nothing under the product package imports oracle/, and bench.py touches it only inside the
    CPU-baseline / reference-arm helpers (oracle_key, cpu_baseline*)."""
    import ast
    import pathlib

    root = pathlib.Path(__file__).resolve().parents[1]

    def oracle_imports(path):
        tree = ast.parse(path.read_text())
        found = []
        for node in ast.walk(tree):
            if isinstance(node, ast.Import) and any(a.name.split(".")[0] == "oracle" for a in node.names):
                found.append(node.lineno)
            if isinstance(node, ast.ImportFrom) and (node.module or "").split(".")[0] == "oracle":
                found.append(node.lineno)
        return found

    for path in (root / "protocols").rglob("*.py"):
        assert oracle_imports(path) == [], f"{path} imports the oracle"
    bench = root / "bench.py"
    tree = ast.parse(bench.read_text())
    allowed = set()
    for node in tree.body:
        if isinstance(node, ast.FunctionDef) and (node.name == "oracle_key" or node.name.startswith("cpu_baseline")):
            allowed.update(range(node.lineno, node.end_lineno + 1))
    assert all(line in allowed for line in oracle_imports(bench)), "bench.py uses the oracle outside the CPU-baseline leg"
