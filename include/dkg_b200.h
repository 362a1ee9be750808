/*
 * dkg_b200 -- C ABI of the B200 batched modular-exponentiation engine for the data-parallel hot
 * path of tno.mpc.protocols.distributed_keygen (threshold Paillier).
 *
 * The reference has no FFI: its hot path is four Python call sites that call third-party
 * pow_mod / mod_inv once per element.  Each entry point below replaces one of those per-element
 * loops by one batched call (reference paths are relative to
 * src/tno/mpc/protocols/distributed_keygen/ in TNO-MPC/protocols.distributed_keygen v4.2.2):
 *
 *   dkg_modexp_batch      <- PaillierSharedKey.partial_decrypt, paillier_shared_key.py:86-93
 *                            (mod_inv when the exponent is negative :89-91, pow_mod :92), looped
 *                            by DistributedPaillier._decrypt_sequence_raw, distributed_keygen.py:463-466;
 *                            also third-party Paillier randomness pow_mod(r, N, N^2)
 *   dkg_combine_batch     <- PaillierSharedKey.decrypt, paillier_shared_key.py:108-125, looped at
 *                            distributed_keygen.py:510-515
 *   dkg_encrypt_batch     <- third-party Paillier.encrypt / randomize: (1 + m N) * r^N mod N^2
 *                            (g = N + 1, distributed_keygen.py:712)
 *   dkg_modexp_grouped    <- DistributedPaillier.__biprime_test_v_calculation,
 *                            distributed_keygen.py:1094,1097, looped by compute_modulus :1313-1329
 *
 * Conventions
 *  - Big integers are arrays of uint32_t limbs, least-significant limb first (the byte order of
 *    int.to_bytes(4*L, "little") and of the reference's key blobs).  A batch is row-major
 *    [count][limbs].
 *  - The caller owns every buffer; nothing is retained after a call returns.
 *  - Functions return DKG_OK or a DKG_ERR_* code; dkg_last_error() gives the text (thread-local).
 *  - Per-element status (uint8_t[count]): DKG_STATUS_OK, DKG_STATUS_NOT_INVERTIBLE (base not a
 *    unit and the exponent is negative: the reference raises ZeroDivisionError from mod_inv),
 *    DKG_STATUS_NOT_DIVISIBLE (combine: (x-1) % N != 0: the reference raises ValueError,
 *    paillier_shared_key.py:119-123).  Rows with a non-zero status are zero-filled.
 *  - Every input value must be < the modulus of its context (the reference's ciphertexts are); a
 *    modexp row that is not gets DKG_STATUS_OUT_OF_RANGE and a zero result instead of a silently
 *    wrong one (the Python-int wrappers reduce first, as the reference's pow_mod does).
 *  - A context is bound to one device and one internal stream; calls on one context serialise.
 *    The *_device variants take device pointers and a cudaStream_t (as void*) and are
 *    asynchronous with respect to the host; everything else is synchronous.
 *  - There is no CPU fallback: without a CUDA device every compute entry point fails with
 *    DKG_ERR_CUDA.
 */
#ifndef DKG_B200_H_
#define DKG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DKG_OK 0
#define DKG_ERR_INVALID 1       /* bad argument (null pointer, even modulus, size out of range) */
#define DKG_ERR_CUDA 2          /* CUDA runtime error or no device */
#define DKG_ERR_UNSUPPORTED 3   /* operand wider than the largest compiled kernel shape */
#define DKG_ERR_NOMEM 4
#define DKG_ERR_NOT_IMPLEMENTED 5

#define DKG_STATUS_OK 0
#define DKG_STATUS_NOT_INVERTIBLE 1
#define DKG_STATUS_NOT_DIVISIBLE 2
#define DKG_STATUS_OUT_OF_RANGE 3   /* modexp: the row is not below the modulus (the result row is zero) */

#define DKG_MAX_LIMBS 272 /* widest modulus the compiled kernel shapes cover (8704 bits) */

typedef struct dkg_modexp_ctx dkg_modexp_ctx;
typedef struct dkg_combine_ctx dkg_combine_ctx;

/* library / device */
int dkg_version(void);
const char* dkg_last_error(void);
int dkg_device_count(int* count);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
unsigned long long dkg_launch_count(void);

/* Process-wide settings (initialised from the environment when first needed, never re-read):
 *   "coop_max"         largest batch a fixed-modulus N^2 context created FROM NOW ON routes to the
 *                      cooperative warp-per-ciphertext kernels (csrc/dkg_coop.cuh), the latency path
 *                      of PaillierSharedKey.partial_decrypt on one / a few ciphertexts
 *                      (distributed_keygen.py:314-382); 0 disables it.  Environment: DKG_COOP_MAX,
 *                      DKG_COOP=0.
 *   "coop_grouped_max" same for the grouped (biprimality) entry points, per call.  Environment:
 *                      DKG_COOP_GROUPED_MAX.
 *   "ct_table"         1: constant-time table access -- every window multiplication reads the
 *                      whole window table (and the Montgomery one) under a mask, so no memory
 *                      address and no branch depends on a digit of the exponent (DESIGN.md §2.11).
 *                      A fixed-exponent context (dkg_modexp_ctx_create, the threshold context)
 *                      takes the setting when it is created; dkg_modexp_grouped and
 *                      dkg_biprime_v_batch read it on every call.  Default 0.  Environment:
 *                      DKG_CT_TABLE=1.
 *   "time_kernels"     see dkg_kernel_times below. */
int dkg_config_set(const char* key, long value);
int dkg_config_get(const char* key, long* value);
/* With dkg_config_set("time_kernels", 1) every launch of an exponentiation kernel of the pair
 * arithmetic (modexp_nsq_kernel, modexp_nsq_multi_kernel) is bracketed by CUDA events on its
 * stream; this call waits for the recorded launches of `device`, returns their durations
 * (milliseconds, in launch order, at most `capacity`) and forgets them. */
int dkg_kernel_times(int device, double* ms, int capacity, int* count);

/* Register-resident mad.wide.u32 microbenchmark: wide multiply-accumulates per second of the
 * integer multiplier on `device`, plain (no carry) and carry-chained.  The roofline denominator. */
int dkg_measure_imad_peak(int device, double* plain_wide_mac_per_s, double* carry_wide_mac_per_s);

/* ---- fixed modulus, fixed signed exponent (per key) --------------------------------------- */
/* modulus: odd, mod_limbs limbs (<= DKG_MAX_LIMBS); exponent: magnitude in exp_limbs limbs,
 * sign in exp_negative (0/1).  Precomputes -N^-1, R mod N, R^2 mod N and the operation list of
 * the exponent (one list for the whole batch: the exponent belongs to the key).  Default: fixed
 * windows, every window multiplies, so the sequence of operations is independent of the exponent's
 * bits (only the table index depends on them); environment DKG_SLIDING_WINDOW=1 selects sliding
 * windows (fewer multiplications, exponent-dependent schedule, as mpz_powm). */
int dkg_modexp_ctx_create(int device, const uint32_t* modulus, int mod_limbs,
                          const uint32_t* exponent, int exp_limbs, int exp_negative,
                          dkg_modexp_ctx** out);
/* Same, for the modulus N^2 given its root n (the Paillier case: partial decryption and encryption
 * randomness work modulo N^2 with N public).  Rows are values modulo N^2 (limbs of N^2, see
 * dkg_modexp_ctx_info / the caller's own count); results are identical to the generic context,
 * the exponentiation runs in pair arithmetic modulo N (csrc/dkg_nsq.cuh). */
int dkg_modexp_ctx_create_nsq(int device, const uint32_t* n, int n_limbs, const uint32_t* exponent,
                              int exp_limbs, int exp_negative, dkg_modexp_ctx** out);
void dkg_modexp_ctx_destroy(dkg_modexp_ctx* ctx);
/* info[0]=K, [1]=M, [2]=padded limbs, [3]=window bits w, [4]=windows (multiplications in the main
 * loop), [5]=exponent bits,
 * [6]=warps per CTA, [7]=CTAs, [8]=1 if the pair arithmetic modulo the root is active,
 * [9]=its K, [10]=its M, [11]=its warps per CTA */
int dkg_modexp_ctx_info(const dkg_modexp_ctx* ctx, int info[12]);

/* out[i] = bases[i] ^ (+-exponent) mod modulus; rows of mod_limbs limbs.  Host buffers. */
int dkg_modexp_batch(dkg_modexp_ctx* ctx, const uint32_t* bases, uint32_t* out, uint8_t* status,
                     size_t count);
/* Same with device buffers on `stream` (cudaStream_t); returns after enqueueing. */
int dkg_modexp_batch_device(dkg_modexp_ctx* ctx, const uint32_t* d_bases, uint32_t* d_out,
                            uint8_t* d_status, size_t count, void* stream);

/* ---- share combination ---------------------------------------------------------------------- */
/* n: the Paillier modulus N (n_limbs limbs); theta_inv: theta^-1 mod N (n_limbs limbs);
 * shares: d+1, the number of partial decryptions multiplied together. */
int dkg_combine_ctx_create(int device, const uint32_t* n, int n_limbs, const uint32_t* theta_inv,
                           int shares, dkg_combine_ctx** out);
void dkg_combine_ctx_destroy(dkg_combine_ctx* ctx);
/* partials: [shares][count][n2_limbs] with n2_limbs = limbs of N^2 (dkg_combine_n2_limbs);
 * out: [count][n_limbs]; status[count]. */
int dkg_combine_n2_limbs(const dkg_combine_ctx* ctx);
int dkg_combine_batch(dkg_combine_ctx* ctx, const uint32_t* partials, uint32_t* out,
                      uint8_t* status, size_t count);
int dkg_combine_batch_device(dkg_combine_ctx* ctx, const uint32_t* d_partials, uint32_t* d_out,
                             uint8_t* d_status, size_t count, void* stream);

/* ---- in-process threshold decryption, sharded by index over the GPUs of one box ------------------ */
/* All d+1 parties' keys in one process (DistributedPaillier with distributed=False: the reference's
 * test / benchmark set-up, distributed_keygen.py:203-226): the two loops of _decrypt_sequence_raw
 * (:463-466 partial decryptions, :510-515 combinations) for every party in one call.  devices: the
 * GPUs to shard over (one host thread + two streams each; rows [count*r/ndev, count*(r+1)/ndev) go to
 * device r; results land in disjoint slices of the caller's arrays; no inter-GPU collective).
 * exponents: [shares][exp_limbs] magnitudes, negative[shares] their signs (party p+1 at index p,
 * paillier_shared_key.py:70-85).  Buffers may be pageable; page-locked ones (dkg_host_register) copy
 * at full PCIe rate. */
typedef struct dkg_threshold_ctx dkg_threshold_ctx;
int dkg_threshold_ctx_create(const int* devices, int ndev, const uint32_t* n, int n_limbs,
                             const uint32_t* theta_inv, int shares, const uint32_t* exponents,
                             int exp_limbs, const uint8_t* negative, dkg_threshold_ctx** out);
void dkg_threshold_ctx_destroy(dkg_threshold_ctx* ctx);
/* info[0]=devices, [1]=shares, [2]=limbs of N, [3]=limbs of N^2 */
int dkg_threshold_info(const dkg_threshold_ctx* ctx, int info[4]);
/* info[0]=1 if the parties share one squaring chain (see below), [1]=its window bits, [2]=its windows,
 * [3],[4]=block size / block count of the pair kernel, [5]=warps per CTA, [6]=CTAs, [7]=rows per chunk */
int dkg_threshold_info_ex(const dkg_threshold_ctx* ctx, int info[8]);
/* ciphertexts [count][n2_limbs] -> plaintexts [count][n_limbs]; the ciphertexts are uploaded once,
 * the partial decryptions stay on the device unless `partials` ([shares][count][n2_limbs]) is given.
 * status[count] (or NULL): the first party's non-zero modexp status, else the combination's. */
int dkg_threshold_decrypt_batch(dkg_threshold_ctx* ctx, const uint32_t* ciphertexts,
                                uint32_t* plaintexts, uint32_t* partials, uint8_t* status, size_t count);
/* The same with everything resident on the context's first device, enqueued on `stream` (a
 * cudaStream_t), no copies: d_partials [shares][count][n2_limbs] and d_status [(shares+1)][count]
 * (every party's modexp status, then the combination's) are required work areas / outputs.
 * With two or more parties whose keys use the pair arithmetic, the d+1 exponentiations of a batch
 * share ONE chain of squarings (right-to-left bucket method, csrc/dkg_nsq.cuh): every partial
 * decryption is still produced, bit-identical to the party's own call.  DKG_SHARED_SQUARINGS=0
 * turns that off (one left-to-right exponentiation per party). */
int dkg_threshold_decrypt_batch_device(dkg_threshold_ctx* ctx, const uint32_t* d_ciphertexts,
                                       uint32_t* d_plaintexts, uint32_t* d_partials,
                                       uint8_t* d_status, size_t count, void* stream);
/* every party's partial decryptions of the same ciphertexts, no combination (loop 1 of
 * _decrypt_sequence_raw, :463-466, for all in-process parties at once; they share one squaring
 * chain like the call above): partials [shares][count][n2_limbs], status [shares][count] or NULL */
int dkg_threshold_partials_batch(dkg_threshold_ctx* ctx, const uint32_t* ciphertexts, uint32_t* partials,
                                 uint8_t* status, size_t count);
/* one party's partial decryptions (what a distributed party computes for its broadcast) */
int dkg_threshold_partial_decrypt_batch(dkg_threshold_ctx* ctx, int party, const uint32_t* ciphertexts,
                                        uint32_t* out, uint8_t* status, size_t count);
/* combination of received partials [shares][count][n2_limbs] */
int dkg_threshold_combine_batch(dkg_threshold_ctx* ctx, const uint32_t* partials, uint32_t* plaintexts,
                                uint8_t* status, size_t count);
/* cudaHostRegister / cudaHostUnregister of a caller buffer (portable across the devices) */
int dkg_host_register(void* ptr, size_t bytes);
int dkg_host_unregister(void* ptr);

/* ---- encryption: (1 + m N) * r^N mod N^2 ---------------------------------------------------- */
/* ctx: a modexp context created with modulus = N^2 and exponent = N.  r: [count][n_limbs],
 * m: [count][n_limbs] or NULL (randomness r^N only); out: [count][n2_limbs]. */
int dkg_encrypt_batch(dkg_modexp_ctx* ctx, const uint32_t* n, int n_limbs, const uint32_t* r,
                      const uint32_t* m, uint32_t* out, size_t count);

/* ---- grouped modexp: per-group modulus and exponent (biprimality test) ----------------------- */
/* moduli: [groups][limbs] (odd); exps: [groups][exp_limbs]; bases: [groups][per_group][limbs];
 * out: same shape as bases.  Montgomery constants are derived on the device per group. */
int dkg_modexp_grouped(int device, const uint32_t* moduli, const uint32_t* exps, int exp_limbs,
                       const uint32_t* bases, uint32_t* out, size_t groups, int per_group,
                       int limbs);

/* ---- the filters around the biprimality test (SURVEY.md section 8f) ---------------------------- */
/* One compute_modulus round's v calculation in one call (distributed_keygen.py:1084-1097):
 * Jacobi symbol of each of the g_per_candidate jointly drawn g's (sympy.jacobi_symbol at :1089),
 * the first `correct` with symbol +1 are raised to exps[g] modulo moduli[g].
 * gvals: [groups][g_per_candidate][limbs]; out_v: [groups][correct][limbs] (rows beyond
 * out_count[g] are zero); out_count[g] = number of usable g's found (<= correct). */
int dkg_biprime_v_batch(int device, const uint32_t* moduli, const uint32_t* exps, int exp_limbs,
                        const uint32_t* gvals, int g_per_candidate, int correct, uint32_t* out_v,
                        int32_t* out_count, size_t groups, int limbs);
/* sym[g][k] = Jacobi symbol (gvals[g][k] / moduli[g]) in {-1, 0, +1}. */
int dkg_jacobi_batch(int device, const uint32_t* moduli, const uint32_t* gvals, int per_group,
                     int8_t* sym, size_t groups, int limbs);
/* flags[g] = 1 if moduli[g] is divisible by one of primes[0..nprimes)
 * (__small_prime_divisors_test, distributed_keygen.py:1197-1209). */
int dkg_small_prime_sieve(int device, const uint32_t* moduli, const uint32_t* primes, int nprimes,
                          uint8_t* flags, size_t groups, int limbs);

/* Biprimality verdict (__biprime_test_with_v_i, distributed_keygen.py:1110-1175) for the in-process
 * case where all parties' v values are at hand: v: [parties][groups][correct][limbs], party 1
 * first; ok[g] = 1 iff every test k < correct has v_1 = +- prod_{i>1} v_i (mod moduli[g]). */
int dkg_biprime_verdict(int device, const uint32_t* moduli, const uint32_t* v, int parties, int correct,
                        uint8_t* ok, size_t groups, int limbs);

/* ---- wire format of the batched partial-decryption message (host only, no device work) ------- */
/* The reference broadcasts {"content": "partial_decryption_sequence", "value": [int, ...]}
 * (distributed_keygen.py:476-484) and reads it back at :497-505.  These two convert between limb
 * rows and the msgpack array that is the "value": integers >= 2^64 as the reference's serializer
 * tags them, {"type": "int", "data": little-endian two's complement of (bits+8)/8 bytes}, smaller
 * ones as minimal native msgpack integers.
 * encode: out == NULL queries the size; *written = bytes needed / written.
 * decode: rows == NULL queries the element count; *consumed = bytes of buf the array occupied;
 * DKG_ERR_INVALID for a negative value, one wider than `limbs`, or malformed input. */
int dkg_wire_encode_rows(const uint32_t* rows, size_t count, int limbs, uint8_t* out,
                         size_t capacity, size_t* written);
int dkg_wire_decode_rows(const uint8_t* buf, size_t len, int limbs, uint32_t* rows,
                         size_t capacity_rows, size_t* count_out, size_t* consumed);

#ifdef __cplusplus
}
#endif
#endif /* DKG_B200_H_ */
