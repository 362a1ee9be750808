"""Constant-time table access (config "ct_table", DESIGN.md §2.11) on every route where the exponent
is secret: the direct kernel of generic contexts, its predicated redo on the pair route, both grouped
(biprimality) kernels and the threshold context's per-party fallback.  Each against CPython pow,
the recorded reference values, or the same computation with the setting off."""
from __future__ import annotations

import math
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _h(x: str) -> int:
    return int(x, 16)


@pytest.fixture()
def ct():
    from protocols.distributed_keygen_b200 import _native

    saved = {k: _native.config_get(k) for k in ("ct_table", "coop_max", "coop_grouped_max")}
    _native.config_set("ct_table", 1)
    yield _native
    for k, v in saved.items():
        _native.config_set(k, v)


def _ct_window(ebits: int, max_w: int = 7) -> int:
    """The window the host picks in constant-time mode (ct_window_cost in csrc/dkg_engine.cu); a
    context that reports it was made in that mode, i.e. runs the constant-time kernels."""
    cost = [(1 << w) - 2 + -(-ebits // w) * (1 + 0.034 * (1 << w)) for w in range(1, max_w + 1)]
    return 1 + min(range(max_w), key=lambda i: (cost[i], i))


def _with_zero_digits(rng: random.Random, bits: int) -> int:
    e = rng.getrandbits(bits) | (1 << (bits - 1))
    # runs of zero bits make whole zero windows at any width up to 7 (the Montgomery-one entry)
    return e & ~(0xFFFFF << (bits // 3)) & ~(0xFFFF << (2 * bits // 3))


@pytest.mark.parametrize("bits", [67, 515, 2051, 4100])
def test_direct_kernel_generic_context(ct, bits):
    from protocols.distributed_keygen_b200 import ModexpContext

    rng = random.Random(bits)
    m = rng.getrandbits(bits) | 1 | (1 << (bits - 1))
    for sign in (1, -1):
        e = sign * _with_zero_digits(rng, bits + 90)
        bases = [v for v in (rng.randrange(1, m) for _ in range(70)) if math.gcd(v, m) == 1]
        ctx = ModexpContext(m, e)
        assert ctx.info()["pair_arithmetic"] == 0
        assert ctx.info()["window_bits"] == _ct_window(abs(e).bit_length())
        assert ctx.modexp(bases) == [pow(b, e, m) for b in bases], (bits, sign)
        ctx.close()


def test_direct_redo_of_the_pair_route(ct):
    """N^2 context, negative exponent, batch above coop_max: a non-unit in the batch makes the
    batched inversion flag it and the whole batch is redone on the direct kernel, in CT mode."""
    from protocols.distributed_keygen_b200 import ModexpContext
    from protocols.distributed_keygen_b200.limbs import ints_to_limbs, limbs_to_ints

    ct.config_set("coop_max", 0)
    rng = random.Random(17)
    p = rng.getrandbits(515) | 1 | (1 << 514)
    q = rng.getrandbits(516) | 1 | (1 << 515)
    n = p * q
    n2 = n * n
    e = -_with_zero_digits(rng, 2 * 1031 + 40)
    vals = []
    while len(vals) < 300:   # (p and q are not primes: draw units)
        v = rng.randrange(1, n2)
        if math.gcd(v, n) == 1:
            vals.append(v)
    bad = {5: 0, 77: n, 150: p * 12345, 233: q, 299: n2 + 5}
    for i, v in bad.items():
        vals[i] = v
    ctx = ModexpContext(n2, e, root=n)
    assert ctx.info()["pair_arithmetic"] == 1
    assert ctx.info()["window_bits"] == _ct_window(abs(e).bit_length()) == 4
    out, status = ctx.modexp_limbs(ints_to_limbs(vals, ctx.limbs))
    ctx.close()
    got = limbs_to_ints(out)
    for i, v in enumerate(vals):
        if i in bad:
            assert status[i] == (3 if v >= n2 else 1) and got[i] == 0, (i, status[i])
        else:
            assert status[i] == 0 and got[i] == pow(v, e, n2), i


def _grouped_cases(rng: random.Random):
    for bits, groups, per_group in [(67, 5, 3), (130, 9, 40), (515, 4, 40), (2050, 3, 40), (2048, 2, 7), (4100, 1, 33)]:
        moduli = [rng.getrandbits(bits) | 1 | (1 << (bits - 1)) for _ in range(groups)]
        exps = [rng.getrandbits(rng.choice([bits - 3, bits // 2, 5])) for _ in range(groups)]
        exps[0] = 0
        if groups > 1:
            exps[1] = _with_zero_digits(rng, bits - 3)
        bases = [[rng.randrange(m) for _ in range(per_group if g % 2 == 0 else max(1, per_group - 2))]
                 for g, m in enumerate(moduli)]
        bases[0][0] = 0
        bases[-1][0] = 0
        yield bits, moduli, exps, bases


@pytest.mark.parametrize("kernel", ["cooperative", "wave"])
def test_grouped_kernels(ct, kernel):
    import protocols.distributed_keygen_b200 as eng

    if kernel == "wave":
        ct.config_set("coop_grouped_max", 0)
    else:
        ct.config_set("coop_grouped_max", 16384)
    rng = random.Random(41)
    for bits, moduli, exps, bases in _grouped_cases(rng):
        got = eng.modexp_grouped(moduli, exps, bases)
        want = [[pow(b, e, m) for b in bs] for m, e, bs in zip(moduli, exps, bases)]
        assert got == want, (kernel, bits)


@pytest.mark.parametrize("kernel", ["cooperative", "wave"])
def test_biprime_v_recorded_values(ct, kernel, biprime_vectors):
    from protocols.distributed_keygen_b200 import distributed_keygen as dkg

    ct.config_set("coop_grouped_max", 16384 if kernel == "cooperative" else 0)
    cases = biprime_vectors["cases"]
    for party in (1, 2, 3):
        mine = [c for c in cases if party <= c["parties"]]
        for correct in sorted({c["correct_param_biprime"] for c in mine}):
            sel = [c for c in mine if c["correct_param_biprime"] == correct]
            batch = [([_h(g) for g in c["g_values"]], _h(c["n"]), _h(c["p_shares"][party - 1]), _h(c["q_shares"][party - 1]))
                     for c in sel]
            got = dkg.biprime_test_v_calculation_batch(batch, party, correct)
            assert got == [[_h(v) for v in c["v"][str(party)]] for c in sel], (kernel, party, correct)


def test_threshold_context_negative_party_and_non_unit(ct):
    """The threshold context falls back to per-party kernels in CT mode: with a party whose exponent
    is negative and a non-unit ciphertext in a batch above coop_max, partials, status and plaintexts
    equal those of the same context with the setting off."""
    from oracle import keys as okeys
    from oracle.paillier_oracle import encrypt_raw
    from protocols.distributed_keygen_b200 import IntegerShares, PaillierSharedKey
    from protocols.distributed_keygen_b200 import distributed_keygen as dkg
    from protocols.distributed_keygen_b200.limbs import ints_to_limbs, limbs_to_ints

    dk = okeys.dealer_keygen(512, 3, 1, seed=4242)
    assert any(k.partial_decrypt_exponent() < 0 for k in dk.keys.values()), "key set without a negative party"
    keys = {}
    for pid, k in dk.keys.items():
        share = IntegerShares(dict(k.share.shares), k.share.degree, k.share.scaling, k.share.number_of_parties)
        keys[pid] = PaillierSharedKey(k.n, k.t, pid, share, k.theta)
    rng = random.Random(8)
    ms = [rng.randrange(dk.n) for _ in range(200)]
    cts = [encrypt_raw(dk.n, m, rng.randrange(1, dk.n)) for m in ms]
    cts[13] = dk.n   # not a unit modulo N^2
    rows = ints_to_limbs(cts, ((dk.n * dk.n).bit_length() + 31) // 32)
    ct.config_set("coop_max", 0)
    res = {}
    for setting in (1, 0):
        ct.config_set("ct_table", setting)
        tctx = dkg.threshold_context(keys, [0])
        parts, pstatus = tctx.partials_limbs(rows)
        plain, status, _ = tctx.decrypt_limbs(rows)
        tctx.close()
        res[setting] = (parts, pstatus, plain, status)
    for a, b in zip(res[1], res[0]):
        assert np.array_equal(a, b)
    plain = limbs_to_ints(res[1][2])
    assert all(plain[i] == m for i, m in enumerate(ms) if i != 13)
    for pid, key in dk.keys.items():
        got = limbs_to_ints(res[1][0][pid - 1])
        assert all(got[i] == key.partial_decrypt(c) for i, c in enumerate(cts) if i != 13), pid
