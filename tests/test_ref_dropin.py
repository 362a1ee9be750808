"""
The drop-in (``protocols.distributed_keygen_b200.patch``) exercised by the REFERENCE's own code:
``DistributedPaillier.decrypt`` / ``_decrypt_raw`` (``distributed_keygen.py:289-382``),
``decrypt_sequence`` / ``_decrypt_sequence_raw`` (``:400-517``) and the name-mangled
``__biprime_test_v_calculation`` (``:1056-1108``) run unmodified on the reference's 24 stored-key
fixtures with the plaintexts of the reference's tests (``test/test_distributed_keygen.py:21-23,
161-185``), parties connected by an in-process pool (tests/ref_harness.py).

* not-gpu part: the patch module imports, binds against the (shimmed) reference and restores it;
  the plumbing is run end to end with the engine twin replaced by the CPU oracle (test double --
  the product has no such path).
* gpu part: the same scenarios with the real engine; every partial decryption and plaintext must
  equal what the unpatched reference computes on the same ciphertexts.
"""
from __future__ import annotations

import random

import pytest

import ref_harness as rh

REF = rh.import_reference()
needs_ref = pytest.mark.skipif(REF is None, reason="no copy of the reference reachable (baseline/_ref or $DKG_REFERENCE_SRC)")

PLAINTEXTS = [1, 2, 3, -1, -2, -3, 1.5, 42.42424242, -1.5, -42.42424242]   # ref: test_distributed_keygen.py:21-23


def _h(x: str) -> int:
    return int(x, 16)


def _sets(fixture_vectors):
    return [(s["t"], s["parties"], s["keys"]) for s in fixture_vectors["sets"]]


def _encrypt_all(n: int, seed: int) -> list[int]:
    from oracle.paillier_oracle import encrypt_raw   # checker-side ciphertext generator

    rng = random.Random(seed)
    return [encrypt_raw(n, rh.encode(m, n), rng.randrange(1, n)) for m in PLAINTEXTS]


def _scenario(schemes, raws):
    """What the reference's tests do: every party decrypts each ciphertext (single) and the whole
    list (sequence); returns (singles[party][i], sequences[party][i], partials[party][i])."""
    parties = sorted(schemes)
    n = schemes[parties[0]].public_key.n
    cts = {p: [rh.ciphertext(schemes[p], c) for c in raws] for p in parties}
    partials = {p: [int(schemes[p].secret_key.partial_decrypt(ct)) for ct in cts[p]] for p in parties}
    singles = {p: [] for p in parties}
    for i in range(len(raws)):
        res = rh.run([schemes[p].decrypt(cts[p][i], apply_encoding=False) for p in parties])
        for p, v in zip(parties, res):
            singles[p].append(int(v))
    res = rh.run([schemes[p].decrypt_sequence(cts[p], apply_encoding=False) for p in parties])
    sequences = {p: [int(v) for v in r] for p, r in zip(parties, res)}
    for p in parties:
        assert [rh.decode(v, n) for v in sequences[p]] == PLAINTEXTS
        assert singles[p] == sequences[p]
    return singles, sequences, partials


@needs_ref
def test_patch_binds_and_restores():
    from protocols.distributed_keygen_b200 import patch

    key_cls, scheme_cls = REF.PaillierSharedKey, REF.DistributedPaillier
    before = (key_cls.partial_decrypt, key_cls.decrypt, scheme_cls._decrypt_sequence_raw,
              scheme_cls.__dict__["_DistributedPaillier__biprime_test_v_calculation"])
    patch.install(REF)
    try:
        assert patch.installed()
        assert key_cls.partial_decrypt is not before[0] and key_cls.decrypt is not before[1]
        assert scheme_cls._decrypt_sequence_raw is not before[2]
        assert hasattr(key_cls, "partial_decrypt_batch") and hasattr(key_cls, "decrypt_batch")
        assert hasattr(scheme_cls, "_b200_biprime_v_batch")
    finally:
        patch.uninstall()
    after = (key_cls.partial_decrypt, key_cls.decrypt, scheme_cls._decrypt_sequence_raw,
             scheme_cls.__dict__["_DistributedPaillier__biprime_test_v_calculation"])
    assert before == after and not hasattr(key_cls, "partial_decrypt_batch")
    assert not patch.install_from_env(REF)   # default: off


@needs_ref
def test_patch_error_behaviour_without_device(fixture_vectors):
    """Type / key checks of paillier_shared_key.py:62-68 are kept; no silent CPU path exists."""
    from protocols.distributed_keygen_b200 import _native, patch

    t, parties, keys = _sets(fixture_vectors)[0]
    schemes = rh.make_schemes(REF, keys, t)
    other = rh.make_schemes(REF, _sets(fixture_vectors)[1][2], _sets(fixture_vectors)[1][0])
    patch.install(REF)
    try:
        key = schemes[1].secret_key
        with pytest.raises(TypeError):
            key.partial_decrypt(12345)
        with pytest.raises(ValueError):
            key.partial_decrypt(rh.ciphertext(other[1], 5))
        if _native.device_count() == 0:
            with pytest.raises(_native.DkgError):
                key.partial_decrypt(rh.ciphertext(schemes[1], 5))
    finally:
        patch.uninstall()


@needs_ref
def test_reference_runs_through_patch_with_engine_double(fixture_vectors, monkeypatch):
    """Plumbing on CPU: reference coroutines + patch + a test double of the engine twin (oracle)."""
    from oracle import paillier_oracle as po
    from protocols.distributed_keygen_b200 import paillier_shared_key as psk
    from protocols.distributed_keygen_b200 import patch

    def fake_partial(self, ciphertexts):
        e = self.partial_decrypt_exponent()
        return [pow(self._raw_value(c), e, self.n_square) for c in ciphertexts]

    def fake_decrypt(self, dicts):
        okey = po.SharedKeyOracle(self.n, self.t, self.player_id, self.share, self.theta)
        return [okey.decrypt(dict(d)) for d in dicts]

    monkeypatch.setattr(psk.PaillierSharedKey, "partial_decrypt_batch", fake_partial)
    monkeypatch.setattr(psk.PaillierSharedKey, "decrypt_batch", fake_decrypt)
    for t, parties, keys in _sets(fixture_vectors):
        n = _h(keys[0]["n"])
        raws = _encrypt_all(n, 1000 + 10 * t + parties)
        plain = _scenario(rh.make_schemes(REF, keys, t), raws)
        for batched in (True, False):
            patch.install(REF, batched_sequence=batched)
            try:
                patched = _scenario(rh.make_schemes(REF, keys, t), raws)
            finally:
                patch.uninstall()
            assert patched == plain


@needs_ref
@pytest.mark.gpu
def test_reference_decrypt_on_gpu_matches_unpatched_reference(fixture_vectors):
    from protocols.distributed_keygen_b200 import launch_count, patch

    for t, parties, keys in _sets(fixture_vectors):
        n = _h(keys[0]["n"])
        raws = _encrypt_all(n, 2000 + 10 * t + parties)
        plain = _scenario(rh.make_schemes(REF, keys, t), raws)      # reference arithmetic (CPython pow)
        for batched in (True, False):
            before = launch_count()
            patch.install(REF, batched_sequence=batched)
            try:
                patched = _scenario(rh.make_schemes(REF, keys, t), raws)
            finally:
                patch.uninstall()
            assert launch_count() > before, "the patched reference did not launch a kernel"
            assert patched == plain


@needs_ref
@pytest.mark.gpu
def test_reference_sequence_on_gpu_with_encrypt_context(fixture_vectors):
    """decrypt(encrypt(m)) == m with GPU encryption, receivers subset (ref: test :233-277)."""
    from protocols.distributed_keygen_b200 import EncryptContext, patch

    t, parties, keys = _sets(fixture_vectors)[-1]
    n = _h(keys[0]["n"])
    rng = random.Random(5)
    enc = EncryptContext(n)
    raws = enc.encrypt([rh.encode(m, n) for m in PLAINTEXTS], [rng.randrange(1, n) for _ in PLAINTEXTS])
    enc.close()
    patch.install(REF)
    try:
        schemes = rh.make_schemes(REF, keys, t)
        ps = sorted(schemes)
        cts = {p: [rh.ciphertext(schemes[p], c) for c in raws] for p in ps}
        names = {p: f"local{p}" for p in ps}
        # only party 1 receives: the others get None (distributed_keygen.py:441-457, 516)
        res = rh.run([
            schemes[p].decrypt_sequence(cts[p], apply_encoding=False,
                                        receivers=["self"] if p == 1 else [names[1]])
            for p in ps
        ])
    finally:
        patch.uninstall()
    assert [rh.decode(int(v), n) for v in res[0]] == PLAINTEXTS
    assert all(r is None for r in res[1:])


@needs_ref
@pytest.mark.gpu
def test_in_process_parties_share_one_engine_call(fixture_vectors, monkeypatch):
    """The reference's in-process parties decrypt the same sequence: once all of them are known to the
    patch, ONE engine call (shared squaring chain) serves every party's ``partial_decrypt_batch`` --
    with exactly the partials each party's own call returns (``DKG_B200_SHARE=0``)."""
    from protocols.distributed_keygen_b200 import EncryptContext, engine, patch

    t, parties, keys = _sets(fixture_vectors)[0]
    n = _h(keys[0]["n"])
    rng = random.Random(11)
    count = 1200
    ms = [rng.randrange(0, 1000) for _ in range(count)]
    enc = EncryptContext(n)
    raws = enc.encrypt([m % n for m in ms], [rng.randrange(1, n) for _ in ms])
    enc.close()
    monkeypatch.setenv("DKG_B200_SHARE_MIN", "1000")
    calls = []
    real = engine.ThresholdContext.partials_limbs
    monkeypatch.setattr(engine.ThresholdContext, "partials_limbs", lambda self, rows: (calls.append(len(rows)), real(self, rows))[1])

    def run_once(share: str):
        monkeypatch.setenv("DKG_B200_SHARE", share)
        patch.install(REF)
        try:
            schemes = rh.make_schemes(REF, keys, t)
            ps = sorted(schemes)
            out = []
            for _ in range(2):          # the first pass makes every party's key known, the second shares
                cts = {p: [rh.ciphertext(schemes[p], c) for c in raws] for p in ps}
                partials = {p: schemes[p].secret_key.partial_decrypt_batch(cts[p]) for p in ps}
                cts = {p: [rh.ciphertext(schemes[p], c) for c in raws] for p in ps}
                res = rh.run([schemes[p].decrypt_sequence(cts[p], apply_encoding=False) for p in ps])
                out.append((partials, [[int(v) for v in r] for r in res]))
            return out
        finally:
            patch.uninstall()

    shared = run_once("1")
    n_shared_calls = len(calls)
    own = run_once("0")
    assert len(calls) == n_shared_calls, "DKG_B200_SHARE=0 must not use the shared call"
    assert n_shared_calls >= 2 and n_shared_calls <= 5, n_shared_calls
    assert shared == own
    for partials, plains in shared:
        assert all(p == ms for p in plains)


def _v_inputs(case):
    return ([_h(g) for g in case["g_values"]], _h(case["n"]), [_h(x) for x in case["p_shares"]],
            [_h(x) for x in case["q_shares"]], case["correct_param_biprime"])


@needs_ref
@pytest.mark.gpu
def test_reference_biprime_v_calculation_on_gpu(biprime_vectors):
    from protocols.distributed_keygen_b200 import patch

    name = "_DistributedPaillier__biprime_test_v_calculation"
    for case in biprime_vectors["cases"]:
        g, n, ps, qs, correct = _v_inputs(case)
        for i in range(1, case["parties"] + 1):
            want = [_h(v) for v in case["v"][str(i)]]
            if len(want) < correct:
                continue   # the reference itself raises on set_share for too few usable g's
            ref_b = getattr(REF.DistributedPaillier, name)(g, i, n, ps[i - 1], qs[i - 1], correct)
            patch.install(REF)
            try:
                got_b = getattr(REF.DistributedPaillier, name)(g, i, n, ps[i - 1], qs[i - 1], correct)
                batch = REF.DistributedPaillier._b200_biprime_v_batch(
                    [(g, n, None, ps[i - 1], qs[i - 1])] * 3, i, correct)
            finally:
                patch.uninstall()
            assert type(got_b) is type(ref_b)
            assert [int(x) for x in got_b.get_share(i)] == [int(x) for x in ref_b.get_share(i)] == want
            assert all([int(x) for x in b.get_share(i)] == want for b in batch)
