#!/usr/bin/env python
"""Cost of constant-time table access (config "ct_table", DESIGN.md §2.11): the same calls with the
setting off and on, alternated in one process, outputs compared between the two and spot-checked
against CPython pow.  One JSON line per case, with the GPU's name and power limit.

Cases: the biprimality batch (2050-bit candidates x 40 bases; 1 and 64 candidates take the
cooperative grouped kernel, 1024 and 16384 the wave kernel), a direct-kernel batch (4102-bit
modulus, 4190-bit exponent) and one party's partial decryptions on the pair kernel.

    python tests/tools/ct_ab.py [--reps 3] [--quick]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402
import protocols.distributed_keygen_b200 as eng  # noqa: E402
from protocols.distributed_keygen_b200 import _native  # noqa: E402
from protocols.distributed_keygen_b200.limbs import ints_to_limbs, limbs_to_ints  # noqa: E402


def gpu_info() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, check=True).stdout.splitlines()[0]
        name, power = (f.strip() for f in out.split(","))
        return {"gpu": name, "power_limit": power}
    except (OSError, subprocess.CalledProcessError, IndexError, ValueError):
        import torch

        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown"}


def ab(label: str, make_call, reps: int, info: dict, extra: dict) -> None:
    """make_call(ct) -> (call, check): call() runs the timed work and returns its output."""
    times = {0: [], 1: []}
    outs = {}
    for ct in (0, 1):   # warm-up, and the outputs compared
        _native.config_set("ct_table", ct)
        call, check = make_call(ct)
        outs[ct] = call()
        check(outs[ct])
    for r in range(reps):
        for ct in ((0, 1) if r % 2 == 0 else (1, 0)):
            _native.config_set("ct_table", ct)
            call, _ = make_call(ct)
            t0 = time.perf_counter()
            call()
            times[ct].append(time.perf_counter() - t0)
    _native.config_set("ct_table", 0)
    same = all(np.array_equal(a, b) for a, b in zip(outs[0], outs[1]))
    off, on = float(np.median(times[0])), float(np.median(times[1]))
    print(json.dumps({"case": label, **extra, "ct_off_ms": round(off * 1e3, 3), "ct_on_ms": round(on * 1e3, 3),
                      "ct_on_over_off": round(on / off, 3), "off_ms_all": [round(t * 1e3, 2) for t in times[0]],
                      "on_ms_all": [round(t * 1e3, 2) for t in times[1]], "outputs_identical": same, **info}), flush=True)
    assert same, label


def grouped_case(C: int, reps: int, info: dict) -> None:
    rng = random.Random(5)
    base_c = min(C, 64)
    moduli, exps = [], []
    for _ in range(base_c):
        ps = [(rng.getrandbits(1024) | (1 << 1023) | 3) if i == 0 else ((rng.getrandbits(1024) | (1 << 1023)) & ~3) for i in range(3)]
        qs = [(rng.getrandbits(1024) | (1 << 1023) | 3) if i == 0 else ((rng.getrandbits(1024) | (1 << 1023)) & ~3) for i in range(3)]
        n = sum(ps) * sum(qs)
        moduli.append(n)
        exps.append((n - ps[0] - qs[0] + 1) // 4)
    L = 65
    reps_c = -(-C // base_c)
    m_arr = np.tile(ints_to_limbs(moduli, L), (reps_c, 1))[:C]
    e_arr = np.tile(ints_to_limbs(exps, L), (reps_c, 1))[:C]
    bases = bench.random_units(C * 40, 1 << 2049, L, 11).reshape(C, 40, L)

    def check(out):
        res = out[0]
        for c, k in ((0, 0), (C // 2, 17), (C - 1, 39)):
            b0 = limbs_to_ints(bases[c, k:k + 1])[0]
            assert limbs_to_ints(res[c, k:k + 1])[0] == pow(b0, exps[c % base_c], moduli[c % base_c])

    def make_call(ct):
        return (lambda: (eng.modexp_grouped_limbs(m_arr, e_arr, bases),)), check

    kernel = "coop_grouped_kernel" if C * 40 <= _native.config_get("coop_grouped_max") else "modexp_grouped_kernel"
    ab("grouped 2050-bit x 40 bases", make_call, reps, info, {"candidates": C, "modexps": 40 * C, "kernel": kernel})


def fixed_case(label: str, modulus: int, exponent: int, root: int | None, count: int, reps: int, info: dict, extra: dict) -> None:
    limbs = (modulus.bit_length() + 31) // 32
    rows = bench.random_units(count, modulus, limbs, 7)
    sample = limbs_to_ints(rows[:2])
    saved = _native.config_get("coop_max")
    _native.config_set("coop_max", 0)
    ctxs = {}
    for ct in (0, 1):   # a context takes the setting when it is created
        _native.config_set("ct_table", ct)
        ctxs[ct] = eng.ModexpContext(modulus, exponent, root=root)
    windows = {("ct_on" if ct else "ct_off"): c.info()["window_bits"] for ct, c in ctxs.items()}

    def check(out):
        assert limbs_to_ints(out[0][:2]) == [pow(b, exponent, modulus) for b in sample], label

    def make_call(ct):
        ctx = ctxs[ct]
        return (lambda: ctx.modexp_limbs(rows)), check

    try:
        ab(label, make_call, reps, info, {"rows": count, **extra, "window_bits": windows})
    finally:
        _native.config_set("coop_max", saved)
        for c in ctxs.values():
            c.close()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes only (a functional run)")
    args = ap.parse_args()
    info = gpu_info()
    saved = _native.config_get("ct_table")
    try:
        for C in ((1, 64) if args.quick else (1, 64, 1024, 16384)):
            grouped_case(C, args.reps, info)
        rng = random.Random(3)
        m = rng.getrandbits(4102) | 1 | (1 << 4101)
        e = rng.getrandbits(4190) | (1 << 4189)
        fixed_case("direct kernel 4102-bit modulus, 4190-bit exponent", m, e, None, 512 if args.quick else 16384,
                   args.reps, info, {"kernel": "modexp_fixed_kernel"})
        half = 1025
        p = rng.getrandbits(half) | 1 | (1 << (half - 1))
        q = rng.getrandbits(half) | 1 | (1 << (half - 1))
        n = p * q
        e = rng.getrandbits(4196) | (1 << 4195)
        fixed_case("one party's partial decryptions, 2050-bit N", n * n, e, n, 1024 if args.quick else 65536,
                   args.reps, info, {"kernel": "modexp_nsq_kernel"})
    finally:
        _native.config_set("ct_table", saved)


if __name__ == "__main__":
    main()
