#!/usr/bin/env python
"""
Benchmark of the threshold-Paillier hot path on B200 (BASELINE.json metric: threshold
decrypts/sec at 2048-bit N).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl reference] [--dump-outputs DIR]
    python bench.py --split --gpus N [--config cfg2|cfg3] [--total T]   # ONE process, one fixed batch
                                                                        # sharded over N GPUs (strong scaling)

Workload (BASELINE.json configs[1]): 3 parties, corruption threshold t=1, key_length 2048
(exact 2048-bit N, 4096-bit N^2; synthetic dealer-generated key and uniformly random ciphertext
units): one *step* = one batch of B ciphertexts per GPU taken through the whole decryption:
d+1 = 3 partial decryptions  c^(e_i) mod N^2  (signed ~4190-bit per-key exponents, one of them
negative => batched modular inversion) + one share combination  (prod mod N^2, L-function,
* theta^-1 mod N).  All d+1 partials are materialised, as they are API-visible values in the
reference (paillier_shared_key.py:52-127, distributed_keygen.py:430-517).

Printed JSON line (rank 0): `value` = threshold decrypts/s with inputs resident in HBM, `e2e` =
the same through the public host-buffer call a user makes (`ThresholdContext.decrypt_limbs` = C ABI
dkg_threshold_decrypt_batch: ciphertexts uploaded ONCE from pinned host memory, d+1 partial
decryptions + combination on the device, plaintexts and all partials read back, inside the timed
region), `e2e.python_int_api` = the same through Python ints, `roofline` = the modexp kernel against
the measured integer-multiplier peak, `cpu_baseline` = GMP mpz_powm (the function gmpy2.powmod
wraps) on all host cores, `latency` = ms per call at B = 1 / 32 / 1024 / 16384 (cooperative
warp-per-ciphertext kernels) next to GMP, `secondary` = the other BASELINE.json configurations.
Multi-GPU: one process per GPU (torchrun), ciphertext batches sharded by index, no data-path
collective; only a barrier and a max-over-ranks of the elapsed time go through NCCL.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "threshold decrypts/sec (2048-bit N)"
UNIT = "decrypts/s"
KEY_NAME = "cfg2_k2048_p3_t1_exact"
WORKLOAD = "cfg2: 3 parties t=1 key_length=2048 (exact 2048-bit N): 3 partial decryptions + share combination per ciphertext"


def shared_config(dk) -> dict:
    """The `config` object both arms print (the driver compares them)."""
    return {"workload": WORKLOAD, "parties": dk.parties, "threshold": dk.t, "modulus_bits": dk.n.bit_length(),
            "key": KEY_NAME}


class KeyData:
    """The synthetic dealer key of the workload (tests/golden/dealer_vectors.json), as plain integers:
    n, parties, t, theta and one Shamir share of lambda*beta per party."""

    def __init__(self, d: dict) -> None:
        self.json = d
        self.n = int(d["n"], 16)
        self.parties = int(d["parties"])
        self.t = int(d["t"])
        self.theta = int(d["theta"], 16)
        self.shares = {int(i): int(v, 16) for i, v in d["shares"].items()}


def load_key() -> KeyData:
    with open(os.path.join(ROOT, "tests", "golden", "dealer_vectors.json")) as fh:
        data = json.load(fh)
    return KeyData(data["keys"][KEY_NAME]["key"])


def oracle_key(dk: KeyData):
    """The oracle's view of the same key: only the CPU-baseline / reference arm may use it."""
    from oracle import keys as okeys

    return okeys.dealer_key_from_json(dk.json)


def hbm_side(traffic_bytes: float, launch_ms: float) -> dict:
    """DRAM bytes of one launch / its duration against the measured copy bandwidth of this pool's
    B200s (MEASURED_PEAKS.json, driver-written; fallback: the profiling recipe's 6.5 TB/s)."""
    peak, src = 6500.0, "fallback 6.5 TB/s (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peak, src = float(json.load(fh)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    achieved = traffic_bytes / (launch_ms * 1e-3) / 1e9
    return {"achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": src}


# DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum) of one launch of the shared-chain
# kernel on 113 664 ciphertexts x 3 parties, from the committed capture (profiles/); None until captured
MULTI_TRAFFIC_113664 = 381.6e9   # 166.0 GB read + 215.6 GB written (profiles/r02_ncu_multi_traffic.csv)


def multi_traffic(B: int):
    return None if MULTI_TRAFFIC_113664 is None else MULTI_TRAFFIC_113664 * B / 113664.0


def canonical_modexp_macs(exp_bits: int, limbs: int) -> float:
    """SURVEY.md section 8(d): modmul(L) = 2L^2 + L wide-MACs; modexp(E, L) = (E + ceil(E/5) + 32)
    modmuls (squarings counted as multiplies, canonical window 5)."""
    return float(exp_bits + (exp_bits + 4) // 5 + 32) * float(2 * limbs * limbs + limbs)


def actual_modexp_macs(info: dict) -> float:
    """Wide multiply-accumulates the kernels really execute per exponentiation (block products of
    K x K limbs, low-half quotient products), from the context's shape and window parameters."""
    # `windows` multiplications in the main loop (the first one is a table load), two domain
    # conversions, one squaring per exponent bit below the first window (bounded by the bit length);
    # table: 2^w - 2 multiplications (fixed windows, the default), or one squaring and 2^(w-1) - 1
    # multiplications for the odd powers (DKG_SLIDING_WINDOW=1)
    w, nd = info["window_bits"], info["windows"]
    sliding = os.environ.get("DKG_SLIDING_WINDOW", "0") not in ("", "0")
    n_sqr = max(info["exponent_bits"] - 1, 0) + (1 if sliding else 0)
    n_mul = max(nd - 1, 0) + (((1 << (w - 1)) - 1) if sliding else ((1 << w) - 2)) + 2
    if info.get("pair_arithmetic"):
        K, M = info["pair_K"], info["pair_M"]
        blk, lo = K * K, K * (K + 1) // 2
        sqr = (M * (M + 1) // 2 + M * M) * blk + M * lo + 2 * M * M * blk + M * lo   # SQR(a) + 2ab
        mul = 3 * M * M * blk + M * lo + 2 * M * M * blk + M * lo                    # ad+bc, ac
    else:
        K, M = info["K"], info["M"]
        blk, lo = K * K, K * (K + 1) // 2
        sqr = (M * (M + 1) // 2 + M * M) * blk + M * lo
        mul = 2 * M * M * blk + M * lo
    return float(n_sqr * sqr + n_mul * mul)


def pair_op_macs(K: int, M: int) -> tuple[float, float]:
    """Wide multiply-accumulates of one squaring / one multiplication in the pair arithmetic modulo N
    with M blocks of K limbs (csrc/dkg_nsq.cuh): (SQR(a) + doubled product, ad+bc + ac)."""
    blk, lo = K * K, K * (K + 1) // 2
    sqr = (M * (M + 1) // 2 + M * M) * blk + M * lo + 2 * M * M * blk + M * lo
    mul = 3 * M * M * blk + M * lo + 2 * M * M * blk + M * lo
    return float(sqr), float(mul)


def shared_chain_macs(info_ex: list, shares: int) -> float:
    """Wide multiply-accumulates the shared-squaring-chain kernel executes per CIPHERTEXT (all
    `shares` partial decryptions): w (nwin - 1) squarings, and per party nwin bucket multiplications
    + 2 (2^w - 2) for folding the buckets + 1 to leave the Montgomery domain; 1 to enter it."""
    _, w, nwin, K, M = info_ex[:5]
    sqr, mul = pair_op_macs(K, M)
    return w * (nwin - 1) * sqr + (1 + shares * (nwin + 2 * ((1 << w) - 2) + 1)) * mul


def threshold_info_ex(tctx) -> list:
    import ctypes

    from protocols.distributed_keygen_b200 import _native

    arr = (ctypes.c_int * 8)()
    _native.check(_native.lib.dkg_threshold_info_ex(tctx._h, ctypes.byref(arr)))
    return list(arr)


def random_units(count: int, n_square: int, limbs: int, seed: int):
    """Uniform random residues below N^2 as limb rows (non-units have negligible probability)."""
    import numpy as np

    rng = np.random.default_rng(seed)
    arr = rng.integers(0, 2**32, size=(count, limbs), dtype=np.uint32)
    top_bits = n_square.bit_length() - 32 * (limbs - 1)
    # clear the top bit of N^2's width so every value is < 2^(bits-1) <= N^2
    arr[:, -1] &= np.uint32((1 << (top_bits - 1)) - 1)
    arr[:, 0] |= np.uint32(1)
    return arr


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int) -> None:
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self) -> None:
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu_index), "-lms", "200"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL,
            )
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        clocks, reasons, mx, power = [], set(), None, []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    clocks.append(float(f[1])); mx = float(f[2]); power.append(float(f[3]))
                except ValueError:
                    continue
                for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if clocks:
            clocks.sort()
            out.update(sm_mhz=clocks[len(clocks) // 2], sm_max_mhz=mx, reasons=sorted(reasons),
                       samples=len(clocks), power_w_max=max(power) if power else None)
        return out


DUMP_ROWS = 8192   # ciphertexts --dump-outputs writes: 3 x 8192 x 128 partial limbs + plaintexts = 30 MB as float64


def dump_outputs(out_dir: str, partials, plaintexts, status) -> None:
    """What the timed call returned in its last step, as float64 arrays of the 32-bit limb values
    (exact): partials [shares, rows, n2_limbs], plaintexts [rows, n_limbs] and status [shares + 1,
    rows] (per party, then the combination; 0 = ok), for a fixed seeded sample of the batch (all of
    it up to DUMP_ROWS ciphertexts) whose row indices go to rows.npy."""
    import numpy as np

    B = plaintexts.shape[0]
    rows = np.arange(B) if B <= DUMP_ROWS else np.sort(np.random.default_rng(2024).choice(B, DUMP_ROWS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in (("rows", rows), ("partials", partials[:, rows]), ("plaintexts", plaintexts[rows]),
                      ("status", status[:, rows])):
        np.save(os.path.join(out_dir, name + ".npy"), arr.astype(np.float64))


def cpu_baseline(dk, cores: int, sample: int, seed: int, cpython: bool = True) -> dict:
    """GMP mpz_powm (+ mpz_invert for the negative exponent) on `cores` pthreads over `sample`
    ciphertexts for each of the d+1 parties, plus the combination in CPython ints: the
    reference's CPU path with the [gmpy] extra (gmpy2.powmod wraps mpz_powm)."""
    from oracle import gmp

    dk = oracle_key(dk)
    n2 = dk.n * dk.n
    limbs = (n2.bit_length() + 31) // 32
    cts = random_units(sample, n2, limbs, seed)
    mod = gmp.int_to_limbs(n2, limbs)
    t0 = time.perf_counter()
    partial_rows = {}
    for pid in range(1, 2 * dk.t + 2):
        e = dk.keys[pid].partial_decrypt_exponent()
        el = gmp.int_to_limbs(abs(e), (abs(e).bit_length() + 31) // 32)
        out, _ = gmp.powm_batch_threads(cts, mod, el, e < 0, cores)
        partial_rows[pid] = gmp.limbs_to_ints(out)
    key1 = dk.keys[1]
    for i in range(sample):
        key1.decrypt({pid: partial_rows[pid][i] for pid in partial_rows})
    secs = time.perf_counter() - t0
    # secondary line: CPython pow on one core (the reference without its [gmpy] extra)
    out = {
        "value": sample / secs, "unit": UNIT, "cores": cores, "kind": "port", "secs": secs,
        "sample": f"{sample} ciphertexts x 3 parties GMP 6.3 mpz_powm/mpz_invert via oracle/c/gmp_batch.c on {cores} pthreads + CPython combine, {secs:.1f} s",
    }
    if cpython:
        k = min(4, sample)
        ints = gmp.limbs_to_ints(cts[:k])
        t1 = time.perf_counter()
        for pid in partial_rows:
            e = dk.keys[pid].partial_decrypt_exponent()
            for c in ints:
                got = pow(pow(c, -1, n2), -e, n2) if e < 0 else pow(c, e, n2)
            assert got == partial_rows[pid][k - 1], "GMP and CPython disagree"
        py_secs = time.perf_counter() - t1
        out["cpython_pow_1core"] = {"value": k / py_secs, "unit": UNIT,
                                    "sample": f"{k} ciphertexts x 3 parties, builtin pow"}
    return out


def gpu_keys(dk, device: int = 0):
    """The engine-side key objects of parties 1..d+1 for a KeyData."""
    import math

    import protocols.distributed_keygen_b200 as eng

    n_fac = math.factorial(dk.parties)
    out = {}
    for pid in range(1, 2 * dk.t + 2):
        share = eng.IntegerShares({pid: dk.shares[pid]}, 2 * dk.t, n_fac * n_fac, dk.parties)
        out[pid] = eng.PaillierSharedKey(dk.n, dk.t, pid, share, dk.theta, device=device)
    return out


def _best_ms(fn, reps: int) -> float:
    fn()
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best * 1e3


def cpu_baseline_rows(rows, modulus: int, exponent: int, cores: int):
    """GMP mpz_powm (+ mpz_invert) over `rows` on `cores` pthreads: (results, seconds).  CPU-baseline
    leg of the latency block (and its checker)."""
    from oracle import gmp

    L = rows.shape[1]
    mag = abs(exponent)
    return gmp.powm_batch_threads(rows, gmp.int_to_limbs(modulus, L), gmp.int_to_limbs(mag, (mag.bit_length() + 31) // 32),
                                  exponent < 0, cores)


def latency_block(dk, cores: int) -> dict:
    """ms per call (host buffers, copies included) of ONE party's partial decryption as a function of
    the batch size -- the reference decrypts one ciphertext per `_decrypt_raw` call and ten in its own
    sequence test -- next to GMP mpz_powm on all host cores for the same rows.  Small batches take the
    cooperative warp-per-ciphertext kernels (csrc/dkg_coop.cuh), large ones the thread-per-ciphertext
    wave kernels; the switch is automatic."""
    import protocols.distributed_keygen_b200 as eng
    from protocols.distributed_keygen_b200.limbs import limbs_to_ints

    keys = gpu_keys(dk)
    n2 = dk.n * dk.n
    rows_out = []
    exps = {pid: k.partial_decrypt_exponent() for pid, k in keys.items()}
    pid = next((p for p, e in exps.items() if e < 0), 1)   # the costlier sign
    e = exps[pid]
    ctx = keys[pid]._modexp_ctx()
    L2 = ctx.limbs
    for B in (1, 32, 1024, 16384):
        cts = random_units(B, n2, L2, 4000 + B)
        res = [None]

        def call():
            res[0] = ctx.modexp_limbs(cts)

        gpu_ms = _best_ms(call, 3 if B <= 1024 else 2)
        sample = cts[: min(B, 4 * cores)]
        want, secs = cpu_baseline_rows(sample, n2, e, cores)
        assert (res[0][0][: len(sample)] == want).all(), "latency block: GPU and GMP disagree"
        cpu_ms = secs / -(-len(sample) // cores) * -(-B // cores) * 1e3
        rows_out.append({"batch": B, "gpu_ms": round(gpu_ms, 3), "gmp_ms": round(cpu_ms, 3),
                         "gpu_per_s": round(B / gpu_ms * 1e3, 1)})
    # full threshold decryption of ONE ciphertext through the reference-shaped scalar calls
    c = limbs_to_ints(random_units(1, n2, L2, 77))[0]

    def one():
        parts = {p: k.partial_decrypt(c) for p, k in keys.items()}
        # (a random unit is not an encryption: skip the combination's divisibility check)
        return parts

    one_ms = _best_ms(one, 3)
    # ... and through the one-call threshold path (all parties' exponentiations in one cooperative
    # launch, combination on the device)
    from protocols.distributed_keygen_b200 import distributed_keygen as dkgmod

    tctx = dkgmod.threshold_context(keys, [0])
    fused = {}
    for B in (1, 32, 1024):
        cts = random_units(B, n2, L2, 5000 + B)
        fused[str(B)] = round(_best_ms(lambda: tctx.decrypt_limbs(cts, want_partials=True), 3), 3)
    tctx.close()
    for k in keys.values():
        k.close()
    return {"op": "partial_decrypt, party %d (exponent sign %s)" % (pid, "-" if e < 0 else "+"), "cpu_cores": cores,
            "rows": rows_out, "three_partials_one_ciphertext_ms": round(one_ms, 3),
            "threshold_decrypt_call_ms_by_batch": fused,
            "note": "gmp_ms = measured on a sample of min(B, 4*cores) rows with all cores, scaled to ceil(B/cores) rounds"}


def secondary_block(peak_tmacs: float) -> list:
    """The BASELINE.json configurations that are not the headline, one entry each, device-resident
    timing with CUDA events (one launch of one kernel wave unless noted), spot-checked against CPython
    pow.  canonical_frac / executed_frac = canonical (SURVEY 8d) and really executed wide-MACs per
    second over the measured IMAD peak of this run."""
    import random

    import numpy as np
    import torch

    import protocols.distributed_keygen_b200 as eng
    from protocols.distributed_keygen_b200.limbs import ints_to_limbs, limbs_to_ints

    with open(os.path.join(ROOT, "tests", "golden", "dealer_vectors.json")) as fh:
        dv = json.load(fh)["keys"]
    out = []
    stream = torch.cuda.current_stream().cuda_stream

    def time_ctx(label, modulus, exponent, root, waves=1):
        ctx = eng.ModexpContext(modulus, exponent, root=root)
        info = ctx.info()
        B = waves * info["ctas"] * info["warps_per_cta"] * 32
        host = random_units(B, modulus, ctx.limbs, 7)
        d_in = torch.from_numpy(host.view(np.int32)).cuda()
        d_out = torch.empty_like(d_in)
        d_st = torch.empty(B, dtype=torch.uint8, device="cuda")
        ctx.modexp_device(d_in.data_ptr(), d_out.data_ptr(), d_st.data_ptr(), B, stream)   # warm-up (same size: same route)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ctx.modexp_device(d_in.data_ptr(), d_out.data_ptr(), d_st.data_ptr(), B, stream)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        got = d_out[B - 1 :].cpu().numpy().view(np.uint32)
        base = limbs_to_ints(host[B - 1 :])[0]
        assert limbs_to_ints(got)[0] == pow(base, exponent, modulus), label
        ebits = abs(exponent).bit_length()
        canon = B * canonical_modexp_macs(ebits, ctx.limbs) / (ms * 1e-3) / 1e12
        execd = B * actual_modexp_macs(info) / (ms * 1e-3) / 1e12
        ctx.close()
        line = {"config": label, "count": B, "ms": round(ms, 2), "per_s": round(B / ms * 1e3, 1),
                "modulus_bits": modulus.bit_length(), "exponent_bits": ebits * (1 if exponent > 0 else -1),
                "kernel": ("modexp_nsq_kernel<%d,%d>" % (info["pair_K"], info["pair_M"])) if info["pair_arithmetic"]
                else ("modexp_fixed_kernel<%d,%d>" % (info["K"], info["M"])),
                "canonical_frac": round(canon / peak_tmacs, 3), "executed_frac": round(execd / peak_tmacs, 3)}
        out.append(line)
        return line

    # cfg2 with a reference-shaped key (N = 2050..2052 bits, 129-limb N^2)
    real = KeyData(dv["cfg2_k2048_p3_t1_real"]["key"])
    kreal = gpu_keys(real)
    for pid in (1, 2):
        time_ctx(f"cfg2 reference-shaped key, partial decrypt party {pid}", real.n * real.n, kreal[pid].partial_decrypt_exponent(), real.n)
    # cfg3: 5 parties t=2: full threshold decryption (5 partials + combination) and combine-only
    c3 = KeyData(dv["cfg3_k2048_p5_t2_exact"]["key"])
    k3 = gpu_keys(c3)
    ex3 = {p: k.partial_decrypt_exponent() for p, k in k3.items()}
    per = [time_ctx(f"cfg3 (5 parties t=2), partial decrypt party {p}", c3.n * c3.n, ex3[p], c3.n) for p in sorted(ex3)]
    comb = k3[1]._combine_ctx()
    Bc = 1 << 17
    parts = torch.from_numpy(random_units(5 * Bc, c3.n * c3.n, comb.n2_limbs, 3).view(np.int32)).cuda()
    d_o = torch.empty((Bc, comb.n_limbs), dtype=torch.int32, device="cuda")
    d_s = torch.empty(Bc, dtype=torch.uint8, device="cuda")
    comb.combine_device(parts.data_ptr(), d_o.data_ptr(), d_s.data_ptr(), Bc, stream)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    comb.combine_device(parts.data_ptr(), d_o.data_ptr(), d_s.data_ptr(), Bc, stream)
    e1.record()
    torch.cuda.synchronize()
    cms = e0.elapsed_time(e1)
    comb_macs = (4 * (2 * 128 * 128 + 128) + 2 * 64 * 64 + 64) * 1.0
    out.append({"config": "cfg3 combine-only, 5 partials (device-resident)", "count": Bc, "ms": round(cms, 3),
                "per_s": round(Bc / cms * 1e3, 1), "canonical_frac": round(Bc * comb_macs / (cms * 1e-3) / 1e12 / peak_tmacs, 3)})
    # full threshold decryption of cfg3 through the one device-resident call (5 partial decryptions
    # on one shared squaring chain + inversion of the negative parties' results + combination)
    from protocols.distributed_keygen_b200 import _native
    from protocols.distributed_keygen_b200 import distributed_keygen as dkgmod

    t3 = dkgmod.threshold_context(k3, [0])
    ix3 = threshold_info_ex(t3)
    B3 = per[0]["count"]
    host3 = random_units(B3, c3.n * c3.n, t3.n2_limbs, 9)
    d_c3 = torch.from_numpy(host3.view(np.int32)).cuda()
    d_p3 = torch.empty((t3.shares, B3, t3.n2_limbs), dtype=torch.int32, device="cuda")
    d_m3 = torch.empty((B3, t3.n_limbs), dtype=torch.int32, device="cuda")
    d_s3 = torch.empty((t3.shares + 1) * B3, dtype=torch.uint8, device="cuda")

    def call3():
        _native.check(_native.lib.dkg_threshold_decrypt_batch_device(t3._h, d_c3.data_ptr(), d_m3.data_ptr(), d_p3.data_ptr(), d_s3.data_ptr(), B3, stream))

    call3()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    call3()
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1)
    got3 = d_p3[:, B3 - 1].cpu().numpy().view(np.uint32)
    base3 = limbs_to_ints(host3[B3 - 1 :])[0]
    for pi, pid in enumerate(sorted(ex3)):
        assert limbs_to_ints(got3[pi : pi + 1])[0] == pow(base3, ex3[pid], c3.n * c3.n), "cfg3 shared chain"
    t3.close()
    ebits3 = max(abs(e).bit_length() for e in ex3.values())
    out.append({"config": "cfg3 threshold decrypt, one device-resident call (5 partial decryptions%s + combination)"
                          % (" on one shared squaring chain, w=%d" % ix3[1] if ix3[0] else ""),
                "count": B3, "ms": round(step_ms, 2), "per_s": round(B3 / step_ms * 1e3, 1),
                "canonical_frac": round(B3 * 5 * canonical_modexp_macs(ebits3, 128) / (step_ms * 1e-3) / 1e12 / peak_tmacs, 3),
                "executed_frac": round(B3 * shared_chain_macs(ix3, 5) / (step_ms * 1e-3) / 1e12 / peak_tmacs, 3) if ix3[0] else None})
    for k in list(kreal.values()) + list(k3.values()):
        k.close()
    # cfg4: key_length 4096; encryption randomness at 2048 and 4096
    c4 = KeyData(dv["cfg4_k4096_p3_t1_exact"]["key"])
    k4 = gpu_keys(c4)
    time_ctx("cfg4 key_length 4096, partial decrypt party 1", c4.n * c4.n, k4[1].partial_decrypt_exponent(), c4.n)
    time_ctx("cfg4 key_length 4096, r^N", c4.n * c4.n, c4.n, c4.n)
    for k in k4.values():
        k.close()
    c2 = KeyData(dv[KEY_NAME]["key"])
    time_ctx("cfg2 key_length 2048, r^N (encryption randomness)", c2.n * c2.n, c2.n, c2.n)
    # cfg5: biprimality-test batch sweep, host buffers end to end, party 1 exponent, 40 bases per candidate
    rng = random.Random(5)
    sweep = []
    for C in (1, 4, 16, 64, 256, 1024, 4096, 16384, 65536, 131072):
        base_c = min(C, 64)
        moduli, exps = [], []
        for _ in range(base_c):
            ps = [(rng.getrandbits(1024) | (1 << 1023) | 3) if i == 0 else ((rng.getrandbits(1024) | (1 << 1023)) & ~3) for i in range(3)]
            qs = [(rng.getrandbits(1024) | (1 << 1023) | 3) if i == 0 else ((rng.getrandbits(1024) | (1 << 1023)) & ~3) for i in range(3)]
            n = sum(ps) * sum(qs)
            moduli.append(n)
            exps.append((n - ps[0] - qs[0] + 1) // 4)
        L = 65
        reps = -(-C // base_c)
        m_arr = np.tile(ints_to_limbs(moduli, L), (reps, 1))[:C]
        e_arr = np.tile(ints_to_limbs(exps, L), (reps, 1))[:C]
        bases = random_units(C * 40, 1 << 2049, L, 11).reshape(C, 40, L)    # < 2^2048 <= N
        eng.modexp_grouped_limbs(m_arr[:1], e_arr[:1], bases[:1])
        t0 = time.perf_counter()
        res = eng.modexp_grouped_limbs(m_arr, e_arr, bases)
        secs = time.perf_counter() - t0
        b0 = limbs_to_ints(bases[C - 1, 39:40])[0]
        assert limbs_to_ints(res[C - 1, 39:40])[0] == pow(b0, exps[(C - 1) % base_c], moduli[(C - 1) % base_c])
        canon = C * 40 * canonical_modexp_macs(2046, 64) / secs / 1e12
        sweep.append({"candidates": C, "modexps": 40 * C, "ms": round(secs * 1e3, 2), "modexps_per_s": round(40 * C / secs, 1),
                      "canonical_frac": round(canon / peak_tmacs, 3)})
    out.append({"config": "cfg5 biprimality-test v_1 batch, 2050-bit candidates, 40 bases each, host buffers end to end "
                          "(<= 16384 modexps: cooperative kernel, above: thread-per-operand kernel)", "sweep": sweep})
    return out


def run_split(args) -> None:
    """ONE process, ONE fixed batch sharded by index over --gpus devices through the public call
    (C ABI dkg_threshold_*): strong scaling with the host gather, as SURVEY.md section 8(e) and
    BASELINE config 3 ("10M ciphertexts across 8 GPUs") describe.  Host buffers are page-locked."""
    import numpy as np

    import protocols.distributed_keygen_b200 as eng
    from protocols.distributed_keygen_b200 import distributed_keygen as dkgmod
    from protocols.distributed_keygen_b200.limbs import limbs_to_ints

    with open(os.path.join(ROOT, "tests", "golden", "dealer_vectors.json")) as fh:
        dv = json.load(fh)["keys"]
    name = KEY_NAME if args.config == "cfg2" else "cfg3_k2048_p5_t2_exact"
    dk = KeyData(dv[name]["key"])
    devices = list(range(args.gpus))
    keys = gpu_keys(dk)
    ctx = dkgmod.threshold_context(keys, devices)
    info = keys[1]._modexp_ctx().info()
    total = args.total or 2 * len(devices) * info["ctas"] * info["warps_per_cta"] * 32
    n2 = dk.n * dk.n
    cts = random_units(total, n2, ctx.n2_limbs, 4242)
    plain = np.zeros((total, ctx.n_limbs), dtype=np.uint32)
    status = np.zeros(total, dtype=np.uint8)
    from protocols.distributed_keygen_b200 import _native

    lines = {}
    with eng.pinned(cts, plain, status):
        def decrypt():
            _native.check(_native.lib.dkg_threshold_decrypt_batch(ctx._h, cts.ctypes.data, plain.ctypes.data, None, status.ctypes.data, total))

        warm = min(total, 4096 * len(devices))
        _native.check(_native.lib.dkg_threshold_decrypt_batch(ctx._h, cts.ctypes.data, plain.ctypes.data, None, status.ctypes.data, warm))
        launches0 = eng.launch_count()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            decrypt()
        secs = (time.perf_counter() - t0) / args.steps
        launches = eng.launch_count() - launches0
        lines["decrypt"] = secs
    # spot check: partials of a few rows against CPython, plaintext against the combination formula
    theta_inv = pow(dk.theta, -1, dk.n)
    exps = {p: k.partial_decrypt_exponent() for p, k in keys.items()}
    for i in (0, total // 2, total - 1):
        c = limbs_to_ints(cts[i : i + 1])[0]
        x = 1
        for p, e in exps.items():
            x = x * (pow(pow(c, -1, n2), -e, n2) if e < 0 else pow(c, e, n2)) % n2
        want = ((x - 1) // dk.n) * theta_inv % dk.n if (x - 1) % dk.n == 0 else None
        got = limbs_to_ints(plain[i : i + 1])[0]
        assert (want is None and status[i] == 2) or (want == got and status[i] == 0), f"split mode: row {i} differs"
    # combine-only on a slice (partials produced by the per-party call)
    sub = min(total, 1 << 20)
    parts = np.zeros((ctx.shares, sub, ctx.n2_limbs), dtype=np.uint32)
    for p in range(ctx.shares):
        parts[p], _ = ctx.partial_decrypt_limbs(p + 1, cts[:sub])
    plain2 = np.zeros((sub, ctx.n_limbs), dtype=np.uint32)
    st2 = np.zeros(sub, dtype=np.uint8)
    with eng.pinned(parts, plain2, st2):
        _native.check(_native.lib.dkg_threshold_combine_batch(ctx._h, parts.ctypes.data, plain2.ctypes.data, st2.ctypes.data, min(sub, 4096)))
        t0 = time.perf_counter()
        _native.check(_native.lib.dkg_threshold_combine_batch(ctx._h, parts.ctypes.data, plain2.ctypes.data, st2.ctypes.data, sub))
        comb_secs = time.perf_counter() - t0
    assert np.array_equal(plain2, plain[:sub]) and np.array_equal(st2, status[:sub])
    ctx.close()
    line = {
        "metric": METRIC if args.config == "cfg2" else "threshold decrypts/sec (2048-bit N, 5 parties t=2)",
        "value": total / secs, "unit": UNIT, "n_gpus": len(devices), "steps": args.steps, "warmup": 1,
        "ms_per_step": secs * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u32 limbs (exact integer)", "data": "synthetic", "mode": "split: one process, one host array in, host gather out",
        "config": {"workload": ("cfg3: 5 parties t=2 key_length=2048: 5 partial decryptions + share combination per ciphertext"
                                if args.config == "cfg3" else WORKLOAD),
                   "parties": dk.parties, "threshold": dk.t, "modulus_bits": dk.n.bit_length(), "key": name},
        "details": {"ciphertexts": total, "devices": devices, "shares": ctx.shares},
        "e2e": {"value": total / secs, "unit": UNIT, "h2d_bytes_per_step": total * ctx.n2_limbs * 4,
                "d2h_bytes_per_step": total * (ctx.n_limbs * 4 + 1)},
        "combine_only": {"value": sub / comb_secs, "unit": "combines/s", "count": sub,
                         "h2d_bytes": sub * ctx.shares * ctx.n2_limbs * 4, "note": "partials start on the host (page-locked): PCIe-bound"},
        "gpu_launches": int(launches),
    }
    print(json.dumps(line), flush=True)


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dk = load_key()
    cores = os.cpu_count() or 1
    sample = args.ref_sample or max(cores * 96, 256)
    for _ in range(min(args.warmup, 1)):
        cpu_baseline(dk, cores, max(cores, 16), 1, cpython=False)
    vals = []
    for s in range(args.steps):
        vals.append(cpu_baseline(dk, cores, sample, 100 + s, cpython=False))
    secs = sum(v["secs"] for v in vals)
    value = sample * args.steps / secs
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs",
        "data": "synthetic", "config": shared_config(dk), "details": {"sample_per_step": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": vals[-1]["sample"]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=0, help="ciphertexts per GPU per step (0 = two full waves of the modexp kernel)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-sample", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the latency block and the secondary configurations")
    ap.add_argument("--split", action="store_true", help="one process, one fixed batch sharded over --gpus devices (strong scaling)")
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3"], help="--split: which BASELINE.json configuration")
    ap.add_argument("--total", type=int, default=0, help="--split: ciphertexts in the batch (0 = two waves per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last one returned (partials, plaintexts, status of "
                         "a fixed sample of rank 0's ciphertexts) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.split):
        ap.error("--dump-outputs: only the default (device-resident threshold decryption) path writes its outputs")

    if args.impl == "reference":
        run_reference(args)
        return
    if args.split and int(os.environ.get("WORLD_SIZE", "1")) == 1:
        run_split(args)
        return

    import numpy as np
    import torch

    import protocols.distributed_keygen_b200 as eng
    from protocols.distributed_keygen_b200 import _native

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    distributed = world > 1
    torch.cuda.set_device(local_rank)
    if distributed:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    dk = load_key()
    shares = 2 * dk.t + 1
    keys = {}
    import math

    n_fac = math.factorial(dk.parties)
    for pid in range(1, shares + 1):
        share = eng.IntegerShares({pid: dk.shares[pid]}, 2 * dk.t, n_fac * n_fac, dk.parties)
        keys[pid] = eng.PaillierSharedKey(dk.n, dk.t, pid, share, dk.theta, device=local_rank)
    ctxs = {pid: key._modexp_ctx() for pid, key in keys.items()}
    comb = keys[1]._combine_ctx()
    L2, Ln = comb.n2_limbs, comb.n_limbs
    info = ctxs[1].info()
    B = args.batch or 2 * info["ctas"] * info["warps_per_cta"] * 32
    exps = {pid: keys[pid].partial_decrypt_exponent() for pid in keys}

    # ---- inputs: real encryptions are not needed for cost, but the result must be checkable:
    # use c = (1 + m N) * u^N style values?  r^N costs a modexp per element on the host, so take
    # uniformly random units and check partials bit-exactly against CPython pow on a sample, and
    # the combination on true encryptions in a small side batch.
    host_cts = random_units(B, dk.n * dk.n, L2, 1000 + rank)
    pinned_cts = torch.from_numpy(host_cts.view(np.int32)).pin_memory()
    d_cts = pinned_cts.cuda(non_blocking=True)
    d_partials = torch.empty((shares, B, L2), dtype=torch.int32, device="cuda")
    d_plain = torch.empty((B, Ln), dtype=torch.int32, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    # One step = the public device-resident call: all d+1 partial decryptions (ONE squaring chain
    # shared by the parties, csrc/dkg_nsq.cuh modexp_nsq_multi_kernel; DKG_SHARED_SQUARINGS=0: one
    # exponentiation per party) + inversion of the negative party's results + the combination.
    from protocols.distributed_keygen_b200 import distributed_keygen as dkgmod

    dev_ctx = dkgmod.threshold_context(keys, [local_rank])
    info_ex = threshold_info_ex(dev_ctx)
    d_status = torch.empty((shares + 1) * B, dtype=torch.uint8, device="cuda")
    d_pstatus, d_cstatus = d_status[: shares * B].view(shares, B), d_status[shares * B :]

    def device_step(record: bool) -> None:
        _native.check(_native.lib.dkg_threshold_decrypt_batch_device(
            dev_ctx._h, d_cts.data_ptr(), d_plain.data_ptr(), d_partials.data_ptr(), d_status.data_ptr(), B, stream))

    # ---- roofline denominator: measured on this GPU, now -------------------------------------
    import ctypes

    plain, carry = ctypes.c_double(0), ctypes.c_double(0)
    _native.check(_native.lib.dkg_measure_imad_peak(local_rank, ctypes.byref(plain), ctypes.byref(carry)))

    for _ in range(args.warmup):
        device_step(False)
    torch.cuda.synchronize()
    _native.config_set("time_kernels", 1)   # CUDA events around every launch of the exponentiation kernel, on its stream
    _native.kernel_times(local_rank)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = eng.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        device_step(True)
    ev1.record()
    barrier()
    launches = eng.launch_count() - launches0
    kernel_ms = _native.kernel_times(local_rank)
    _native.config_set("time_kernels", 0)
    clocks = sampler.stop() if rank == 0 else {}
    elapsed_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    if distributed:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())

    # ---- parity spot-check of what was just timed, against CPython integers --------------------
    # (the full parity suite against the oracle and the reference's golden vectors is tests/)
    from protocols.distributed_keygen_b200.limbs import limbs_to_ints

    part_host = d_partials.cpu().numpy().view(np.uint32)
    n2 = dk.n * dk.n
    for s, pid in enumerate(range(1, shares + 1)):
        e = exps[pid]
        for i in (0, B // 3, B - 1):
            c = limbs_to_ints(host_cts[i : i + 1])[0]
            want = pow(pow(c, -1, n2), -e, n2) if e < 0 else pow(c, e, n2)
            got = limbs_to_ints(part_host[s, i : i + 1])[0]
            assert got == want, f"rank {rank}: partial decryption mismatch party {pid} element {i}"
    assert int(d_pstatus.max().item()) == 0 and int(d_cstatus.max().item()) == 0

    # ---- the same step WITHOUT the shared squaring chain: one left-to-right exponentiation per party
    # (each party's own call, what separate processes / machines would run) + the combination; one
    # untimed and one timed pass, reported next to `value` so that the share of the speed-up that
    # needs all parties in one process is visible
    per_party_ms = None
    if world == 1 and not args.no_secondary:
        d_parts2 = torch.empty_like(d_partials)
        d_st2 = torch.empty((shares, B), dtype=torch.uint8, device="cuda")
        d_plain2 = torch.empty_like(d_plain)
        d_cst2 = torch.empty(B, dtype=torch.uint8, device="cuda")

        def per_party_step():
            for s_, pid in enumerate(range(1, shares + 1)):
                ctxs[pid].modexp_device(d_cts.data_ptr(), d_parts2[s_].data_ptr(), d_st2[s_].data_ptr(), B, stream)
            comb.combine_device(d_parts2.data_ptr(), d_plain2.data_ptr(), d_cst2.data_ptr(), B, stream)

        per_party_step()
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        per_party_step()
        p1.record()
        torch.cuda.synchronize()
        per_party_ms = p0.elapsed_time(p1)
        assert torch.equal(d_parts2, d_partials) and torch.equal(d_plain2, d_plain), "shared chain and per-party kernels disagree"
        del d_parts2, d_plain2
    plain_host = d_plain.cpu().numpy().view(np.uint32)
    theta_inv = pow(dk.theta, -1, dk.n)
    for i in (0, B // 2, B - 1):
        x = 1
        for s in range(shares):
            x = x * limbs_to_ints(part_host[s, i : i + 1])[0] % n2
        assert (x - 1) % dk.n == 0, "combined value minus one not divisible by N"
        assert limbs_to_ints(plain_host[i : i + 1])[0] == ((x - 1) // dk.n) * theta_inv % dk.n, "combine mismatch"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, part_host, plain_host, d_status.cpu().numpy().reshape(shares + 1, B))

    # ---- end to end through the public host-buffer call ------------------------------------------
    e2e = None
    if not args.no_e2e:
        from protocols.distributed_keygen_b200 import distributed_keygen as dkgmod

        tctx = dev_ctx
        pinned_partials = torch.empty((shares, B, L2), dtype=torch.int32).pin_memory()
        pinned_plain = torch.empty((B, Ln), dtype=torch.int32).pin_memory()
        pinned_status = torch.empty(B, dtype=torch.uint8).pin_memory()
        np_cts = pinned_cts.numpy().view(np.uint32)

        def e2e_step():
            # one call: H2D of the ciphertexts (once), 3 partial decryptions + combination, D2H of
            # the plaintexts, every party's partials and the status bytes
            _native.check(_native.lib.dkg_threshold_decrypt_batch(
                tctx._h, np_cts.ctypes.data, pinned_plain.data_ptr(), pinned_partials.data_ptr(), pinned_status.data_ptr(), B))

        e2e_steps = args.steps
        e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            e2e_step()
        barrier()
        secs = time.perf_counter() - t0
        t = torch.tensor([secs], dtype=torch.float64, device="cuda")
        if distributed:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_secs = float(t.item())
        assert not pinned_status.numpy().any()
        assert np.array_equal(pinned_partials.numpy().view(np.uint32)[:, : min(B, 4096)], part_host[:, : min(B, 4096)])
        assert np.array_equal(pinned_plain.numpy().view(np.uint32), plain_host)
        h2d = B * L2 * 4
        d2h = shares * B * L2 * 4 + B * Ln * 4 + B
        e2e = {"value": world * B * e2e_steps / e2e_secs, "unit": UNIT, "steps": e2e_steps,
               "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h * world,
               "call": "ThresholdContext.decrypt_limbs / dkg_threshold_decrypt_batch (ciphertexts uploaded once; plaintexts + all partials + status read back)"}
        tctx.close()
        if rank == 0:
            # the same through Python ints (the reference-shaped signatures: lists of int in and out)
            k_int = min(B, info["ctas"] * info["warps_per_cta"] * 32)   # one full wave of ciphertexts
            ints = limbs_to_ints(host_cts[:k_int])
            t0 = time.perf_counter()
            got_int = dkgmod.decrypt_sequence_local(keys, ints)
            py_secs = time.perf_counter() - t0
            assert got_int[:8] == limbs_to_ints(plain_host[:8])
            e2e["python_int_api"] = {"value": k_int / py_secs, "unit": UNIT, "batch": k_int,
                                     "call": "distributed_keygen.decrypt_sequence_local (Python ints in, Python ints out, one engine call)"}

    # ---- true encryptions through the same kernels: decrypt(encrypt(m)) == m -------------------
    import random

    def encrypt_raw(n, m, r):  # (1 + m N) * r^N mod N^2, g = N + 1
        return (1 + m * n) * pow(r, n, n * n) % (n * n)

    rng = random.Random(7 + rank)
    ms = [rng.randrange(dk.n) for _ in range(64)]
    cts_small = [encrypt_raw(dk.n, m, rng.randrange(1, dk.n)) for m in ms]
    parts = {pid: keys[pid].partial_decrypt_batch(cts_small) for pid in keys}
    got = keys[1].decrypt_batch([{pid: parts[pid][i] for pid in keys} for i in range(64)])
    assert got == ms, "threshold decryption round trip failed"

    if rank == 0:
        # dominant kernel: its launches were bracketed by CUDA events on their stream inside the timed
        # region (dkg_kernel_times).  Shared chain: ONE launch per step does all `shares`
        # exponentiations of the batch; otherwise one launch per party.
        shared_chain = bool(info_ex[0])
        avg_ms = sum(kernel_ms) / len(kernel_ms)
        assert len(kernel_ms) == args.steps * (1 if shared_chain else shares), "kernel launch count"
        modexps_per_launch = shares if shared_chain else 1
        ebits = sum(abs(exps[pid]).bit_length() for pid in exps) / len(exps)
        macs_per_launch = B * modexps_per_launch * canonical_modexp_macs(int(round(ebits)), L2)
        achieved = macs_per_launch / (avg_ms * 1e-3) / 1e12
        actual = B * (shared_chain_macs(info_ex, shares) if shared_chain else actual_modexp_macs(info)) / (avg_ms * 1e-3) / 1e12
        kname = ("modexp_nsq_multi_kernel<%d,%d>" if shared_chain else "modexp_nsq_kernel<%d,%d>") % (info["pair_K"], info["pair_M"])
        # roofline denominator: the better of the two register-resident IMAD.WIDE probes measured
        # in this run (ptxas issues every IMAD.WIDE at 4-cycle intervals per sub-partition, so both
        # forms top out near 32 wide-MAC/clk/SM = 9.3 T/s at 1965 MHz)
        peak = max(plain.value, carry.value) / 1e12
        value = world * B * args.steps / (max_ms * 1e-3)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": max_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (exact integer)",
            "data": "synthetic",
            "config": shared_config(dk),
            "details": {
                "ciphertexts_per_gpu_per_step": B, "n2_limbs": L2,
                "exponent_bits": [abs(exps[p]).bit_length() * (1 if exps[p] > 0 else -1) for p in sorted(exps)],
                "kernel_shape": info, "parallelism": f"index-sharded x{world}, no collective",
                "cache": "inputs+outputs per step (%.0f MB) larger than L2" % ((shares + 1) * B * L2 * 4 / 1e6),
                "without_shared_squaring_chain": (None if per_party_ms is None else {
                    "value": B / (per_party_ms * 1e-3), "unit": UNIT, "ms_per_step": per_party_ms,
                    "note": "one left-to-right exponentiation per party (every party's own call) + combination, same batch, "
                            "one timed pass; all partials and plaintexts bit-identical to the timed path"}),
            },
            "roofline": {
                "bound": "imad", "achieved": achieved, "peak": peak, "unit": "T wide-MAC/s",
                "frac": achieved / peak,
                # DRAM bytes of one launch of this kernel: ncu dram__bytes_read.sum + dram__bytes_write.sum
                # captured once on a 113 664-ciphertext launch (profiles/r01_ncu_nsq_traffic_final.csv:
                # 37.80 GB + 8.72 GB, window tables spilling out of L2), scaled to this launch's size;
                # only known for the pair-arithmetic kernel at 2048-bit N
                "traffic": multi_traffic(B) if shared_chain else ((46.523e9 * B / 113664.0) if (info.get("pair_arithmetic") and info.get("pair_K") == 14) else None),
                "traffic_unit": "bytes per launch (DRAM, from the committed ncu capture)",
                # the HBM side of the roofline, to show the kernel is nowhere near it
                "hbm": (hbm_side(multi_traffic(B), avg_ms) if (shared_chain and multi_traffic(B)) else
                        hbm_side(46.523e9 * B / 113664.0, avg_ms) if (not shared_chain and info.get("pair_arithmetic") and info.get("pair_K") == 14) else None),
                "kernel": kname, "kernel_share_of_step": avg_ms * len(kernel_ms) / max_ms,
                "modexps_per_launch": B * modexps_per_launch,
                "shared_squaring_chain": ({"window_bits": info_ex[1], "windows": info_ex[2]} if shared_chain else None),
                "actual_wide_mac": actual, "frac_actual": actual / peak,
                "avg_launch_ms": avg_ms, "algorithmic_macs_per_launch": macs_per_launch,
                "peak_source": "dkg_measure_imad_peak, measured in this run: max of register-resident mad.wide.u32 (plain) and mad.lo.cc/madc.hi.cc (carry chain) probes",
                "peak_plain_mad_wide": plain.value / 1e12,
                "peak_carry_chain": carry.value / 1e12,
                "note": "achieved = canonical work of SURVEY 8(d) (2L^2+L per modmul at L=limbs of N^2, squarings as multiplies, one "
                        "independent exponentiation per partial decryption) / the kernel's measured duration; the kernel computes the same "
                        "partial decryptions with fewer multiplies (block squaring; pair arithmetic modulo N; ONE squaring chain shared by "
                        "the parties of a ciphertext, csrc/dkg_nsq.cuh), so achieved/peak exceeds 1; frac_actual = multiplies really "
                        "executed / peak is the pipe-level figure",
            },
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if e2e is not None:
            line["e2e"] = e2e
        cores = os.cpu_count() or 1
        if world == 1:
            line["cpu_baseline"] = cpu_baseline(dk, cores, args.cpu_sample or max(cores * 96, 256), 5)
            if not args.no_secondary:
                for key in keys.values():
                    key.close()
                line["latency"] = latency_block(dk, cores)
                line["secondary"] = secondary_block(peak)
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
