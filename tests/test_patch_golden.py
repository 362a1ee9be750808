"""
The drop-in (``protocols.distributed_keygen_b200.patch``) without a copy of the reference: the patch
is installed on a stand-in of the reference's interface (``tests/ref_standin``, names only, no
arithmetic), and what the patched methods return is compared with what the reference's OWN classes
computed on the same keys and ciphertexts (``tests/golden/fixture_vectors.json``: partial
decryptions and plaintexts of the reference's 24 stored-key fixtures; ``biprime_vectors.json``: its v
values).  ``tests/test_ref_dropin.py`` runs the same patch inside the real reference when a copy of
it is available.

* not-gpu part: binding, restoring, the argument checks that precede any device work, and the
  plumbing with the engine twin replaced by the CPU oracle (test double -- the product has no such
  path).
* gpu part: ``partial_decrypt`` / ``decrypt`` and their batched forms, the batched
  ``_decrypt_sequence_raw`` between in-process parties (also with a subset of receivers), the shared
  engine call of in-process parties, and ``__biprime_test_v_calculation``.
"""
from __future__ import annotations

import random

import pytest

import ref_harness as rh
import ref_standin as REF

V_CALC = "_DistributedPaillier__biprime_test_v_calculation"


def _h(x: str) -> int:
    return int(x, 16)


def _sets(fixture_vectors):
    return [(s["t"], s["keys"], s["vectors"]) for s in fixture_vectors["sets"]]


def _bound():
    return (REF.PaillierSharedKey.partial_decrypt, REF.PaillierSharedKey.decrypt,
            REF.DistributedPaillier._decrypt_sequence_raw, REF.DistributedPaillier.__dict__[V_CALC])


def test_patch_binds_and_restores_on_standin():
    from protocols.distributed_keygen_b200 import patch

    before = _bound()
    for batched in (True, False):
        patch.install(REF, batched_sequence=batched)
        try:
            assert patch.installed()
            now = _bound()
            assert now[0] is not before[0] and now[1] is not before[1] and now[3] is not before[3]
            assert (now[2] is not before[2]) == batched
            assert hasattr(REF.PaillierSharedKey, "partial_decrypt_batch") and hasattr(REF.PaillierSharedKey, "decrypt_batch")
            assert hasattr(REF.DistributedPaillier, "_b200_biprime_v_batch")
        finally:
            patch.uninstall()
        assert _bound() == before and not hasattr(REF.PaillierSharedKey, "partial_decrypt_batch")
    assert not patch.install_from_env(REF)   # default: off


def test_patched_key_checks_its_arguments(fixture_vectors):
    from protocols.distributed_keygen_b200 import _native, patch

    sets = _sets(fixture_vectors)
    schemes = rh.make_schemes(REF, sets[0][1], sets[0][0])
    other = rh.make_schemes(REF, sets[1][1], sets[1][0])
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


def test_patch_plumbing_with_engine_double(fixture_vectors, monkeypatch):
    """Plumbing on CPU: patch + a test double of the engine twin (oracle) reproduce the reference's
    partials and plaintexts through the key methods and the batched sequence decryption."""
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
    patch.install(REF)
    try:
        for t, keys, vectors in _sets(fixture_vectors):
            good = [v for v in vectors if "error" not in v]
            schemes = rh.make_schemes(REF, keys, t)
            for pid, scheme in schemes.items():
                assert [scheme.secret_key.partial_decrypt(rh.ciphertext(scheme, _h(v["c"]))) for v in good] == \
                    [_h(v["partials"][str(pid)]) for v in good]
            ps = sorted(schemes)
            res = rh.run([schemes[p]._decrypt_sequence_raw([rh.ciphertext(schemes[p], _h(v["c"])) for v in good]) for p in ps])
            assert all([int(e.value) for e in r] == [_h(v["plaintext"]) for v in good] for r in res)
    finally:
        patch.uninstall()


@pytest.mark.gpu
def test_patched_key_matches_reference_vectors(fixture_vectors):
    from protocols.distributed_keygen_b200 import launch_count, patch

    before = launch_count()
    patch.install(REF)
    try:
        for t, keys, vectors in _sets(fixture_vectors):
            schemes = rh.make_schemes(REF, keys, t)
            good = [v for v in vectors if "error" not in v]   # the error vector holds a tampered partial
            for pid, scheme in schemes.items():
                key = scheme.secret_key
                cts = [rh.ciphertext(scheme, _h(v["c"])) for v in good]
                want = [_h(v["partials"][str(pid)]) for v in good]
                assert key.partial_decrypt(cts[0]) == want[0]
                assert key.partial_decrypt_batch(cts) == want
            key = schemes[1].secret_key
            dicts = [{int(p): _h(x) for p, x in v["partials"].items()} for v in good]
            assert key.decrypt(dicts[0]) == _h(good[0]["plaintext"])
            assert key.decrypt_batch(dicts) == [_h(v["plaintext"]) for v in good]
            for v in vectors:
                if "error" in v:
                    assert v["error"] == "ValueError"
                    with pytest.raises(ValueError):
                        key.decrypt({int(p): _h(x) for p, x in v["partials"].items()})
    finally:
        patch.uninstall()
    assert launch_count() > before, "the patched methods did not launch a kernel"


@pytest.mark.gpu
def test_patched_decrypt_sequence_matches_reference_vectors(fixture_vectors):
    """The batched ``_decrypt_sequence_raw`` of every in-process party (messages through the
    in-process pool) returns the reference's plaintexts; with ``receivers`` only party 1 gets them."""
    from protocols.distributed_keygen_b200 import patch

    patch.install(REF)
    try:
        for t, keys, vectors in _sets(fixture_vectors):
            good = [v for v in vectors if "error" not in v]
            want = [_h(v["plaintext"]) for v in good]
            schemes = rh.make_schemes(REF, keys, t)
            ps = sorted(schemes)
            res = rh.run([schemes[p]._decrypt_sequence_raw([rh.ciphertext(schemes[p], _h(v["c"])) for v in good]) for p in ps])
            assert all([int(e.value) for e in r] == want for r in res)
            schemes = rh.make_schemes(REF, keys, t)
            res = rh.run([
                schemes[p]._decrypt_sequence_raw([rh.ciphertext(schemes[p], _h(v["c"])) for v in good],
                                                 receivers=["self"] if p == 1 else ["local1"])
                for p in ps
            ])
            assert [int(e.value) for e in res[0]] == want and all(r is None for r in res[1:])
    finally:
        patch.uninstall()


@pytest.mark.gpu
def test_in_process_parties_share_one_engine_call(fixture_vectors, monkeypatch):
    """Once every party's key is known to the patch, ONE engine call (shared squaring chain) serves
    every party's ``partial_decrypt_batch``, with exactly the partials each party's own call returns
    (``DKG_B200_SHARE=0``)."""
    from protocols.distributed_keygen_b200 import EncryptContext, engine, patch

    t, keys, _ = _sets(fixture_vectors)[0]
    n = _h(keys[0]["n"])
    rng = random.Random(11)
    ms = [rng.randrange(0, 1000) for _ in range(1200)]
    enc = EncryptContext(n)
    raws = enc.encrypt(ms, [rng.randrange(1, n) for _ in ms])
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
                partials = {p: schemes[p].secret_key.partial_decrypt_batch([rh.ciphertext(schemes[p], c) for c in raws]) for p in ps}
                res = rh.run([schemes[p]._decrypt_sequence_raw([rh.ciphertext(schemes[p], c) for c in raws]) for p in ps])
                out.append((partials, [[int(e.value) for e in r] for r in res]))
            return out
        finally:
            patch.uninstall()

    shared = run_once("1")
    n_shared_calls = len(calls)
    own = run_once("0")
    assert len(calls) == n_shared_calls, "DKG_B200_SHARE=0 must not use the shared call"
    assert 2 <= n_shared_calls <= 5, n_shared_calls
    assert shared == own
    for _, plains in shared:
        assert all(p == ms for p in plains)


@pytest.mark.gpu
def test_patched_biprime_v_calculation_matches_reference_vectors(biprime_vectors):
    from protocols.distributed_keygen_b200 import patch

    patch.install(REF)
    try:
        checked = 0
        for case in biprime_vectors["cases"]:
            g, n = [_h(x) for x in case["g_values"]], _h(case["n"])
            ps, qs = [_h(x) for x in case["p_shares"]], [_h(x) for x in case["q_shares"]]
            correct = case["correct_param_biprime"]
            for i in range(1, case["parties"] + 1):
                want = [_h(v) for v in case["v"][str(i)]]
                if len(want) < correct:
                    continue   # the reference itself raises on set_share for too few usable g's
                got = getattr(REF.DistributedPaillier, V_CALC)(g, i, n, ps[i - 1], qs[i - 1], correct)
                batch = REF.DistributedPaillier._b200_biprime_v_batch([(g, n, None, ps[i - 1], qs[i - 1])] * 3, i, correct)
                assert got.get_share(i) == want
                assert all(b.get_share(i) == want for b in batch)
                checked += 1
        assert checked > 0
    finally:
        patch.uninstall()
