// C ABI of the engine (include/dkg_b200.h): contexts, constant derivation, kernel dispatch.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/dkg_b200.h"
#include "dkg_host_bigint.h"
#include "dkg_modexp_params.h"
#include "dkg_combine.cuh"
#include "dkg_aux_kernels.cuh"
#include "dkg_grouped_params_fwd.h"
#include "dkg_biprime.cuh"
#include "dkg_nsq_params_fwd.h"
#include "dkg_nsq_io.cuh"
#include "dkg_coop_params.h"
#include "dkg_kernel_table.h"

namespace {

thread_local std::string g_err;
std::atomic<unsigned long long> g_launches{0};

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t e__ = (expr);                                                               \
    if (e__ != cudaSuccess)                                                                 \
      return fail(DKG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__));       \
  } while (0)

// ---- kernel shapes -----------------------------------------------------------------------------
// (K, M): block size and block count; padded width K*M limbs.  Sorted by padded width.
struct Shape { int K, M; };
constexpr Shape kShapes[] = {
    {4, 1},  {4, 2},  {4, 3},   {8, 2},   {6, 3},   {12, 2},  {16, 2},  {12, 3},  {16, 3},
    {16, 4}, {22, 3}, {16, 5},  {16, 6},  {16, 8},  {12, 11}, {16, 9},  {16, 12}, {16, 16},
    {20, 13}, {16, 17},
};

// A CTA-uniform constant in the layout of a lane-private operand ([vector][lane], vectors of
// VW = 4 limbs when K % 4 == 0, else 2): multiplication operands are always read with this
// one stride (see WarpIO in dkg_modexp.cuh), so constants that get multiplied are replicated.
void append_lane_replicated(std::vector<uint32_t>& out, const std::vector<uint32_t>& c, int K) {
  const int VW = (K % 4 == 0) ? 4 : 2;
  for (size_t v = 0; v < c.size() / VW; ++v)
    for (int lane = 0; lane < 32; ++lane)
      for (int e = 0; e < VW; ++e) out.push_back(c[v * VW + e]);
}
}  // namespace
namespace dkg {
void launch_group_setup(const GroupedParams& p, bool ct_table, cudaStream_t stream);
// dkg_coop.cu: the cooperative (warp-per-operand) latency kernels
int coop_max_warps(int K, bool pair_kernel);
cudaError_t launch_coop_nsq(int K, const CoopNsqParams& p, int ctas, int warps, size_t smem, cudaStream_t stream);
cudaError_t launch_coop_grouped(int K, bool ct_table, const CoopGroupedParams& p, int ctas, int warps, size_t smem,
                                cudaStream_t stream);
cudaError_t launch_coop_combine(int K, const CoopCombineParams& p, int ctas, int warps, size_t smem, cudaStream_t stream);
}  // namespace dkg
namespace {

// every kernel compiled for shape (K, M), whichever dkg_kernels_<n>.cu holds it
dkg::ShapeKernels lookup_kernels(int K, int M) {
  dkg::ShapeKernels k;
  for (auto g : {dkg::find_kernels_group0, dkg::find_kernels_group1, dkg::find_kernels_group2,
                 dkg::find_kernels_group3, dkg::find_kernels_group4, dkg::find_kernels_group5})
    g(K, M, &k);
  return k;
}

bool pick_shape(int limbs, Shape* out) {
  for (const Shape& s : kShapes)
    if (s.K * s.M >= limbs) { *out = s; return true; }
  return false;
}

constexpr size_t kMaxDynSmem = 227 * 1024;

struct DeviceState {
  int device = -1;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  uint32_t* scratch = nullptr;
  size_t scratch_words = 0;
  unsigned int* counter = nullptr;
  uint32_t* aux = nullptr;  // batched-inversion buffers
  size_t aux_words = 0;
  cudaEvent_t last = nullptr;  // end of the latest launch sequence that used scratch / aux / counter
  std::mutex mu;            // held while a launch sequence is enqueued (and, for host buffers, until it is done)
  // event pairs around the exponentiation kernels' launches (config "time_kernels"), read and
  // cleared by dkg_kernel_times: the kernel's own duration for the roofline, measured in place
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ktimes;
};
std::atomic<long> g_time_kernels{0};
struct KernelTimer {
  DeviceState* d; cudaStream_t s; cudaEvent_t e0 = nullptr, e1 = nullptr;
  KernelTimer(DeviceState* d_, cudaStream_t s_) : d(d_), s(s_) {
    if (g_time_kernels.load() == 0 || d->ktimes.size() >= 4096) return;
    if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) { e0 = e1 = nullptr; return; }
    cudaEventRecord(e0, s);
  }
  ~KernelTimer() { if (e1) { cudaEventRecord(e1, s); d->ktimes.emplace_back(e0, e1); } }
};

// All contexts of a device share its scratch areas and the work ticket.  Every launch sequence --
// from the host-buffer entry points on the internal stream and from the *_device entry points on
// the caller's stream alike -- is enqueued under the device mutex and ordered on the device after
// the previous one (cudaStreamWaitEvent on `last`), so two streams or threads can never have
// kernels of this library running against the same scratch at the same time.
struct DeviceLease {
  DeviceState* d;
  cudaStream_t s;
  std::unique_lock<std::mutex> lk;
  DeviceLease(DeviceState* d_, cudaStream_t s_) : d(d_), s(s_), lk(d_->mu) {
    cudaSetDevice(d->device);
    cudaStreamWaitEvent(s, d->last, 0);
  }
  ~DeviceLease() { cudaEventRecord(d->last, s); }
};
std::mutex g_dev_mu;
DeviceState g_devs[16];

int device_state(int device, DeviceState** out) {
  if (device < 0 || device >= 16) return fail(DKG_ERR_INVALID, "device index out of range");
  std::lock_guard<std::mutex> lk(g_dev_mu);
  DeviceState& d = g_devs[device];
  if (d.device < 0) {
    int count = 0;
    CUDA_TRY(cudaGetDeviceCount(&count));
    if (device >= count) return fail(DKG_ERR_CUDA, "no such CUDA device");
    CUDA_TRY(cudaSetDevice(device));
    CUDA_TRY(cudaDeviceGetAttribute(&d.sm_count, cudaDevAttrMultiProcessorCount, device));
    CUDA_TRY(cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaMalloc(&d.counter, sizeof(unsigned int)));
    CUDA_TRY(cudaEventCreateWithFlags(&d.last, cudaEventDisableTiming));
    // batch buffers of the host-buffer entry points come from the stream-ordered pool and stay
    // cached there between calls (no cudaMalloc/cudaFree on the data path)
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    d.device = device;
  }
  *out = &d;
  return DKG_OK;
}

int ensure_scratch(DeviceState* d, size_t words) {
  if (d->scratch_words >= words) return DKG_OK;
  CUDA_TRY(cudaSetDevice(d->device));
  if (d->scratch) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaFree(d->scratch));
    d->scratch = nullptr;
    d->scratch_words = 0;
  }
  cudaError_t e = cudaMalloc(&d->scratch, words * sizeof(uint32_t));
  if (e != cudaSuccess) {
    cudaGetLastError();   // (clear it: callers may fall back to a smaller layout and launch again)
    d->scratch = nullptr;
    return fail(DKG_ERR_NOMEM, std::string("scratch cudaMalloc: ") + cudaGetErrorString(e));
  }
  d->scratch_words = words;
  return DKG_OK;
}

struct DevBufs {
  cudaStream_t stream = nullptr;
  std::vector<void*> ptrs;
  explicit DevBufs(cudaStream_t s) : stream(s) {}
  ~DevBufs() { for (void* p : ptrs) if (p) cudaFreeAsync(p, stream); }
  template <typename T> cudaError_t alloc(T** out, size_t bytes) {
    void* p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, bytes ? bytes : 1, stream);
    if (e == cudaSuccess) ptrs.push_back(p);
    *out = (T*)p;
    return e;
  }
};

int ensure_aux(DeviceState* d, size_t words) {
  if (d->aux_words >= words) return DKG_OK;
  CUDA_TRY(cudaSetDevice(d->device));
  if (d->aux) {
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaFree(d->aux));
    d->aux = nullptr;
    d->aux_words = 0;
  }
  cudaError_t e = cudaMalloc(&d->aux, words * sizeof(uint32_t));
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("aux cudaMalloc: ") + cudaGetErrorString(e));
  d->aux_words = words;
  return DKG_OK;
}

}  // namespace


namespace {

// Lane plan of one product phase of the cooperative kernels (transcription of make_plan in
// tests/coop_model.py): diagonal d of an nb x nb block product has the tiles (i, d - i),
// max(0, d - nb + 1) <= i <= min(d, nb - 1); lane d is its primary, spare lanes take further chunks
// of the long diagonals so that no lane has more than `c` tiles, c minimal.
dkg::CoopPlanTable make_coop_plan(int nb, int ndiag) {
  dkg::CoopPlanTable t{};
  for (int l = 0; l < 32; ++l) { t.d[l] = 0; t.i0[l] = 0; t.i1[l] = 0; t.partner[0][l] = t.partner[1][l] = t.partner[2][l] = -1; }
  std::vector<int> lo(ndiag), hi(ndiag), len(ndiag), chunks(ndiag);
  for (int d = 0; d < ndiag; ++d) {
    lo[d] = std::max(0, d - nb + 1);
    hi[d] = std::min(d, nb - 1) + 1;
    len[d] = hi[d] - lo[d];
  }
  int c = 1;
  for (;; ++c) {
    int lanes = 0, most = 0;
    for (int d = 0; d < ndiag; ++d) { const int k = (len[d] + c - 1) / c; lanes += k; most = std::max(most, k); }
    if (lanes <= 32 && most <= 4) break;
  }
  int next = ndiag, rounds = 0;
  for (int d = 0; d < ndiag; ++d) {
    chunks[d] = (len[d] + c - 1) / c;
    const int per = (len[d] + chunks[d] - 1) / chunks[d];
    for (int k = 0; k < chunks[d]; ++k) {
      const int a = lo[d] + k * per, b = std::min(lo[d] + (k + 1) * per, hi[d]);
      const int lane = k == 0 ? d : next++;
      t.d[lane] = (uint8_t)d; t.i0[lane] = (uint8_t)a; t.i1[lane] = (uint8_t)std::max(a, b);
      if (k > 0) t.partner[k - 1][d] = (int8_t)lane;
    }
    rounds = std::max(rounds, chunks[d] - 1);
  }
  t.rounds = rounds;
  t.ndiag = ndiag;
  return t;
}

// block size / block count of the cooperative kernels for `limbs` limbs per number
bool coop_shape(int limbs, int* K, int* nb) {
  for (int k : {6, 12}) {
    const int n = (limbs + k - 1) / k;
    if (n <= dkg::kCoopMaxBlocks) { *K = k; *nb = n; return true; }
  }
  return false;
}

long env_long(const char* name, long dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atol(v) : dflt;
}
// Largest batch the cooperative kernels take (0 disables them): below it a warp per operand beats
// waiting for a thread-per-operand wave (DESIGN.md section 2.10 has the measured crossover).
// Process-wide settings, initialised from the environment once (DKG_COOP=0 disables,
// DKG_COOP_MAX / DKG_COOP_GROUPED_MAX set the limits) and changed through dkg_config_set; a
// fixed-modulus context takes its limit when it is created.
std::atomic<long> g_coop_max{-1}, g_coop_grouped_max{-1}, g_ct_table{-1};
bool ct_table_setting() {
  long v = g_ct_table.load();
  if (v < 0) { v = env_long("DKG_CT_TABLE", 0) != 0 ? 1 : 0; g_ct_table.store(v); }
  return v != 0;
}
size_t coop_limit(std::atomic<long>& slot, const char* env_name, long dflt) {
  long v = slot.load();
  if (v < 0) {
    v = env_long("DKG_COOP", 1) == 0 ? 0 : std::max(0L, env_long(env_name, dflt));
    slot.store(v);
  }
  return (size_t)v;
}
constexpr long kCoopMaxDefault = 16384, kCoopGroupedMaxDefault = 16384;

}  // namespace

struct dkg_modexp_ctx {
  DeviceState* dev = nullptr;
  int limbs = 0;  // caller-visible row width
  Shape shape{};
  int Lp = 0;
  int wbits = 1, nops = 0, tab_entries = 0, nmul = 0, ebits = 0, table_odd = 0;
  int negative = 0;
  uint32_t n0inv = 0;
  int warps = 1, ctas = 1;
  size_t smem = 0;
  size_t scratch_per_warp = 0;
  size_t scratch_q_offset = 0;
  dkg::KernelFn kernel = nullptr;
  dkg::BatchInvFn inv_kernel = nullptr;
  int inv_warps = 1;
  size_t inv_smem = 0;
  uint32_t* d_consts = nullptr;
  uint32_t* d_ops = nullptr;
  // pair arithmetic modulo N when the modulus is N^2 with known N (dkg_nsq.cuh)
  bool nsq = false;
  bool nsq_bg = false;             // b component in global scratch (wide keys: twice the warps per SM)
  bool nsq_inv = false;            // negative exponents inverted inside the pair kernels (pair_invert)
  size_t ninv_slot = 0;            // first spare pair slot of a warp's scratch for that
  Shape nshape{};
  int nLp = 0, nLs = 0, nwarps = 1;   // dense / slot-layout limbs of a pair component
  size_t nsmem = 0, nscratch_per_warp = 0, nscratch_q_offset = 0;
  uint32_t n_n0inv = 0;
  dkg::NsqFn nsq_kernel = nullptr;
  uint32_t* d_nconsts = nullptr;   // kernel constants
  uint32_t* d_nio = nullptr;       // entry/exit constants
  // cooperative (warp-per-operand) latency path for small batches (dkg_coop.cuh): its own R = 2^(32 cLc)
  bool coop = false;
  int cK = 0, cnb = 0, cLc = 0;
  size_t coop_max = 0;             // largest batch routed to it
  uint32_t* d_cconsts = nullptr;   // kernel constants (CoopNsqParams::consts)
  uint32_t* d_cio = nullptr;       // entry/exit constants for cLc
  dkg::CoopPlanTable cfull{}, clow{};
  bool ct_table = false;           // constant-time table access (masked scan of all entries)
};

namespace {

// Window width 1..max_w of least cost(ebits, w), in multiplications (the narrowest on a tie).
int choose_window(int ebits, int max_w, double (*cost)(int ebits, int w)) {
  int best = 1;
  for (int w = 2; w <= max_w; ++w)
    if (cost(ebits, w) < cost(ebits, best)) best = w;
  return best;
}

// Fixed windows: 2^w - 2 multiplications build the table, then one per digit.
double fixed_window_cost(int ebits, int w) { return (double)(((1L << w) - 2) + (ebits + w - 1) / w); }

// Constant-time table access: every multiplication scans all 2^w entries (~0.034 of a
// multiplication's time per entry at 2048-bit N: 560 B per thread against the L2/HBM share of a
// thread), so narrower windows win: cost = 2^w - 2 + ceil(E/w) * (1 + 0.034 * 2^w).
double ct_window_cost(int ebits, int w) {
  return (double)((1L << w) - 2) + (double)((ebits + w - 1) / w) * (1.0 + 0.034 * (double)(1L << w));
}

// Sliding windows for the fixed-exponent contexts.  The exponent belongs to the key, so the whole
// batch shares ONE operation list, built here once: "square nsq times, then multiply by the odd
// power table[idx]".  Table: c^1, c^3, ..., c^(2^w - 1), i.e. 2^(w-1) entries from one squaring and
// 2^(w-1) - 1 multiplications; a window of w bits costs a multiplication only every ~w+1 bits.
// op = (nsq << 8) | idx, idx 0xff = no multiplication (trailing zeros); the first op has nsq = 0
// and means "start from table[idx]".
constexpr uint32_t kOpNoMul = 0xffu;
constexpr uint32_t kOpMulOne = 0xfeu;  // fixed windows: digit 0 multiplies by the Montgomery one
double sliding_window_cost(int ebits, int w) { return (double)((1L << (w - 1)) + ebits / (w + 1)); }
std::vector<uint32_t> sliding_window_ops(const uint32_t* e, int ebits, int w, int* table_entries, int* nmul) {
  auto bit = [&](int i) { return (e[i / 32] >> (i % 32)) & 1u; };
  std::vector<uint32_t> ops;
  int maxidx = -1, muls = 0;
  uint32_t pending = 0;
  int i = ebits - 1;
  while (i >= 0) {
    if (!bit(i)) { ++pending; --i; continue; }
    int l = std::max(i - w + 1, 0);
    while (!bit(l)) ++l;
    uint32_t v = 0;
    for (int b = i; b >= l; --b) v = (v << 1) | bit(b);
    const uint32_t idx = (v - 1) / 2;
    const uint32_t nsq = ops.empty() ? 0u : pending + (uint32_t)(i - l + 1);
    ops.push_back((nsq << 8) | idx);
    maxidx = std::max(maxidx, (int)idx);
    ++muls;
    pending = 0;
    i = l - 1;
  }
  if (pending) ops.push_back((pending << 8) | kOpNoMul);
  *table_entries = maxidx + 1;
  *nmul = muls;
  return ops;
}

// Chain warps of the batched inversion: chains of 32 groups keep the binary-GCD count at 1/32 of
// the elements but leave most SMs idle (56 warps for a 56 832-element launch); the chain products
// dominate, so spread them over every SM as long as a chain keeps at least 4 groups.
int inversion_chain_warps(const DeviceState* d, const dkg_modexp_ctx* ctx, unsigned long long ngroups) {
  unsigned long long nchain = (ngroups + 31) / 32;
  const unsigned long long wide = std::min<unsigned long long>((unsigned long long)d->sm_count * std::max(ctx->inv_warps, 1), ngroups / 4);
  if (wide > nchain) nchain = wide;
  return (int)std::max<unsigned long long>(nchain, 1);
}

// Batched inversion of `count` rows modulo ctx's modulus: Montgomery's trick along chains of ~32
// groups, one binary-GCD inversion per chain lane.  Its work area is the start of d->aux,
//   chain_s | chain_p | scratch | chain_status | any_bad (32 words),
// and callers put their own buffers behind it.  Returns its size in words; with `b`, also lays it
// out there (d->aux must already be that large).
size_t batchinv_area(const dkg_modexp_ctx* ctx, size_t count, dkg::BatchInvParams* b = nullptr) {
  const DeviceState* d = ctx->dev;
  const unsigned long long ngroups = (count + 31) / 32;
  const size_t gwords = (size_t)ctx->Lp * 32;
  const int nchain = inversion_chain_warps(d, ctx, ngroups);
  if (b) {
    b->chain_s = d->aux; b->chain_p = d->aux + ngroups * gwords; b->scratch = d->aux + 2 * ngroups * gwords;
    b->chain_status = b->scratch + (size_t)nchain * gwords;
    b->any_bad = reinterpret_cast<unsigned int*>(b->chain_status + (size_t)nchain * 32);
    b->nchain_warps = nchain; b->chain_len = (int)((ngroups + nchain - 1) / nchain);
  }
  return 2 * ngroups * gwords + (size_t)nchain * gwords + (size_t)nchain * 32 + 32;
}

// Launches the batched inversion of `rows` in the area above.  plain_out null: the inverses stay in
// chain_s (Montgomery form, lane layout) for the direct kernel, which takes *b.  Otherwise they go
// there as canonical rows (`rows` itself is fine: a chain warp reads all its groups before it writes
// any), and *b->any_bad is set on the device if a chain met a non-unit.
int launch_batchinv(dkg_modexp_ctx* ctx, const uint32_t* rows, size_t count, uint32_t* plain_out, cudaStream_t stream,
                    dkg::BatchInvParams* b) {
  *b = dkg::BatchInvParams{};
  batchinv_area(ctx, count, b);
  b->bases = rows; b->count = count; b->in_limbs = ctx->limbs; b->consts = ctx->d_consts; b->n0inv = ctx->n0inv;
  b->plain_out = plain_out;
  if (plain_out) CUDA_TRY(cudaMemsetAsync(b->any_bad, 0, sizeof(unsigned int), stream));
  else b->any_bad = nullptr;
  const int blocks = (b->nchain_warps + ctx->inv_warps - 1) / ctx->inv_warps;
  ctx->inv_kernel<<<blocks, ctx->inv_warps * 32, ctx->inv_smem, stream>>>(*b);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return DKG_OK;
}

// CTAs of a wave launch of ctas x warps warps: fewer when the batch has fewer groups of 32 rows
int wave_ctas(int ctas, int warps, size_t count) {
  const unsigned long long ngroups = (count + 31) / 32;
  return ngroups < (unsigned long long)ctas * warps ? (int)((ngroups + warps - 1) / warps) : ctas;
}

// The direct kernel (dkg_modexp.cuh) on `count` rows.  inv: batched inversion of the bases to take
// instead of inverting each one, or null; run_if: device flag that predicates the launch, or null.
int launch_direct(dkg_modexp_ctx* ctx, const uint32_t* d_bases, uint32_t* d_out, uint8_t* d_status,
                  const uint32_t* d_final_mul, size_t count, cudaStream_t stream, const dkg::BatchInvParams* inv,
                  const unsigned int* run_if) {
  DeviceState* d = ctx->dev;
  int rc = ensure_scratch(d, (size_t)ctx->ctas * ctx->warps * ctx->scratch_per_warp);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), stream));
  dkg::ModexpParams p{};
  if (inv) { p.inv_mont = inv->chain_s; p.chain_status = inv->chain_status; p.nchain_warps = inv->nchain_warps; }
  p.bases = d_bases; p.out = d_out; p.status = d_status; p.count = count; p.in_limbs = ctx->limbs;
  p.consts = ctx->d_consts; p.ops = ctx->d_ops; p.nops = ctx->nops; p.tab_entries = ctx->tab_entries; p.table_odd = ctx->table_odd;
  p.negative = ctx->negative; p.n0inv = ctx->n0inv; p.scratch = d->scratch;
  p.scratch_per_warp = ctx->scratch_per_warp; p.scratch_q_offset = ctx->scratch_q_offset; p.counter = d->counter; p.final_mul = d_final_mul;
  p.run_if = run_if;
  ctx->kernel<<<wave_ctas(ctx->ctas, ctx->warps, count), ctx->warps * 32, ctx->smem, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return DKG_OK;
}

// out-of-range rows (>= modulus) are flagged and zeroed after the compute kernels
int launch_range_check(dkg_modexp_ctx* ctx, const uint32_t* d_bases, uint32_t* d_out, uint8_t* d_status, size_t count,
                       cudaStream_t stream) {
  const unsigned blocks = (unsigned)((count * 32 + 255) / 256);
  dkg::range_check_kernel<<<blocks, 256, 0, stream>>>(d_bases, ctx->d_consts, ctx->limbs, count, d_out, d_status);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return DKG_OK;
}

// Launch geometry of the cooperative kernels: one instance per warp; spread small batches over the
// SMs first (one warp per CTA), then stack warps, then go persistent (work ticket).
void coop_grid(const DeviceState* d, int K, bool pair_kernel, size_t count, int* ctas, int* warps) {
  const int maxw = dkg::coop_max_warps(K, pair_kernel);
  if (count <= (size_t)d->sm_count) { *warps = 1; *ctas = (int)count; return; }
  *warps = (int)std::min<size_t>(maxw, (count + d->sm_count - 1) / d->sm_count);
  *ctas = (int)std::min<size_t>((count + *warps - 1) / *warps, (size_t)d->sm_count * std::max(1, maxw / *warps));
}

// Small batches modulo N^2: entry -> cooperative pair exponentiation (a warp per (party,
// ciphertext), negative exponents inverted in the kernel, per-element status) -> exit.  `parties`
// are contexts of ONE key (same N, hence the same cooperative constants and plans): their partial
// decryptions of the same ciphertexts go out as [nparties][count][limbs] in one launch sequence,
// so that a threshold decryption of a few ciphertexts costs one exponentiation's latency, not d+1.
int launch_modexp_coop_parties(dkg_modexp_ctx* const* parties, int nparties, const uint32_t* d_bases, uint32_t* d_out,
                               uint8_t* d_status, size_t count, cudaStream_t stream, const uint32_t* d_mrows, int m_limbs) {
  dkg_modexp_ctx* ctx = parties[0];
  DeviceState* d = ctx->dev;
  const int Lc = ctx->cLc;
  const size_t instances = count * (size_t)nparties;
  int ctas = 1, warps = 1;
  coop_grid(d, ctx->cK, true, instances, &ctas, &warps);
  size_t per_warp = 0;
  for (int p = 0; p < nparties; ++p) per_warp = std::max(per_warp, ((size_t)parties[p]->tab_entries + 1) * 2 * Lc);
  const size_t pair_words = (count + instances) * (size_t)(2 * Lc);
  int rc = ensure_scratch(d, (size_t)ctas * warps * per_warp);
  if (rc == DKG_OK) rc = ensure_aux(d, pair_words);
  if (rc != DKG_OK) return rc;
  uint32_t* pairs_in = d->aux;
  uint32_t* pairs_out = d->aux + count * (size_t)(2 * Lc);
  dkg::NsqIoParams e{};
  e.in = d_bases; e.out = pairs_in; e.count = count; e.io_limbs = ctx->limbs; e.Lp = Lc; e.consts = ctx->d_cio; e.n0inv = ctx->n_n0inv;
  e.mrows = nullptr; e.m_limbs = 0;
  dkg::nsq_entry_kernel<<<(unsigned)((count + 63) / 64), 64, 0, stream>>>(e);
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), stream));
  dkg::CoopNsqParams q{};
  q.pairs_in = pairs_in; q.pairs_out = pairs_out; q.status = d_status; q.count = count; q.nb = ctx->cnb;
  q.consts = ctx->d_cconsts; q.nparties = nparties;
  for (int p = 0; p < nparties; ++p) {
    q.ops[p] = parties[p]->d_ops; q.nops[p] = parties[p]->nops; q.tab_entries[p] = parties[p]->tab_entries;
    q.table_odd[p] = parties[p]->table_odd; q.negative[p] = parties[p]->negative;
  }
  q.ct_table = ctx->ct_table ? 1 : 0;
  q.scratch = d->scratch; q.scratch_per_warp = per_warp; q.counter = d->counter; q.full = ctx->cfull; q.low = ctx->clow;
  const size_t smem = ((size_t)dkg::kCoopNsqConsts + (size_t)dkg::kCoopNsqWarpBufs * warps) * Lc * 4;
  CUDA_TRY(dkg::launch_coop_nsq(ctx->cK, q, ctas, warps, smem, stream));
  dkg::NsqIoParams x = e;
  x.in = pairs_out; x.out = d_out; x.count = instances; x.mrows = d_mrows; x.m_limbs = m_limbs;
  dkg::nsq_exit_kernel<<<(unsigned)((instances + 63) / 64), 64, 0, stream>>>(x);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(3);
  return DKG_OK;
}

// Modulus N^2 with known N: entry (pairs) -> pair exponentiation -> exit, from `src` (the bases, or
// their batched inversion) through `pairs` (count * 2 nLp words) to d_out.
int launch_pair(dkg_modexp_ctx* ctx, const uint32_t* src, uint32_t* pairs, uint32_t* d_out, uint8_t* d_status,
                size_t count, cudaStream_t stream, const uint32_t* d_mrows, int m_limbs) {
  DeviceState* d = ctx->dev;
  int rc = ensure_scratch(d, (size_t)ctx->ctas * ctx->nwarps * ctx->nscratch_per_warp);
  if (rc != DKG_OK) return rc;
  dkg::NsqIoParams e{};
  e.in = src; e.out = pairs; e.count = count; e.io_limbs = ctx->limbs; e.Lp = ctx->nLp; e.consts = ctx->d_nio; e.n0inv = ctx->n_n0inv;
  e.mrows = nullptr; e.m_limbs = 0;
  dkg::nsq_entry_kernel<<<(unsigned)((count + 63) / 64), 64, 0, stream>>>(e);
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), stream));
  dkg::NsqParams q{};
  q.pairs_in = pairs; q.pairs_out = pairs; q.count = count; q.consts = ctx->d_nconsts; q.ops = ctx->d_ops;
  q.nops = ctx->nops; q.tab_entries = ctx->tab_entries; q.table_odd = ctx->table_odd; q.ct_table = ctx->ct_table ? 1 : 0; q.scratch = d->scratch; q.scratch_per_warp = ctx->nscratch_per_warp;
  q.negative = ctx->negative && ctx->nsq_inv ? 1 : 0; q.status = d_status; q.inv_slot = ctx->ninv_slot;
  if (d_status) CUDA_TRY(cudaMemsetAsync(d_status, 0, count, stream));
  q.scratch_q_offset = ctx->nscratch_q_offset; q.counter = d->counter;
  {
    KernelTimer kt(d, stream);
    ctx->nsq_kernel<<<wave_ctas(ctx->ctas, ctx->nwarps, count), ctx->nwarps * 32, ctx->nsmem, stream>>>(q);
  }
  dkg::NsqIoParams x = e;
  x.in = pairs; x.out = d_out; x.mrows = d_mrows; x.m_limbs = m_limbs;
  dkg::nsq_exit_kernel<<<(unsigned)((count + 63) / 64), 64, 0, stream>>>(x);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(3);
  return DKG_OK;
}

// How one fixed-exponent call runs (pick_route decides from the context and the batch size):
enum class Route {
  coop,       // N^2 context, batch <= coop_max: entry -> cooperative pair kernel -> exit
  pair,       // N^2 context, positive exponent or in-kernel inversion: entry -> pair kernel -> exit
  pair_redo,  // N^2 context, negative exponent: batched inversion -> pair route -> direct kernel if
              // a chain of the inversion met a non-unit, so that the per-element status comes out exact
  direct,     // anything else: [batched inversion ->] direct kernel
};

Route pick_route(const dkg_modexp_ctx* ctx, size_t count) {
  if (!ctx->nsq) return Route::direct;
  if (ctx->coop && count <= ctx->coop_max) return Route::coop;
  if (!ctx->negative || ctx->nsq_inv) return Route::pair;
  return ctx->inv_kernel ? Route::pair_redo : Route::direct;
}

// Encryption's factor (1 + m N): m rows folded into the exit kernel of the pair routes, whole rows
// multiplied in by the direct kernel.
struct EncryptFactor { const uint32_t* m; int m_limbs; const uint32_t* final_mul; };

// One fixed-exponent call on `count` device rows by its route, then the range check (which
// encryption's pair routes skip).
int launch_modexp(dkg_modexp_ctx* ctx, const uint32_t* d_bases, uint32_t* d_out, uint8_t* d_status, size_t count,
                  cudaStream_t stream, const EncryptFactor* enc = nullptr) {
  if (count == 0) return DKG_OK;
  DeviceState* d = ctx->dev;
  CUDA_TRY(cudaSetDevice(d->device));
  const Route route = pick_route(ctx, count);
  const uint32_t* mrows = enc ? enc->m : nullptr;
  const int m_limbs = enc ? enc->m_limbs : 0;
  dkg::BatchInvParams inv{};
  int rc = DKG_OK;
  if (route == Route::coop) {
    rc = launch_modexp_coop_parties(&ctx, 1, d_bases, d_out, d_status, count, stream, mrows, m_limbs);
  } else if (route == Route::direct) {
    const bool batched = ctx->negative && ctx->inv_kernel != nullptr && count > 32;   // >= 2 groups
    if (batched) rc = ensure_aux(d, batchinv_area(ctx, count));
    if (rc == DKG_OK && batched) rc = launch_batchinv(ctx, d_bases, count, nullptr, stream, &inv);
    if (rc == DKG_OK)
      rc = launch_direct(ctx, d_bases, d_out, d_status, enc ? enc->final_mul : nullptr, count, stream, batched ? &inv : nullptr, nullptr);
  } else if (route == Route::pair) {
    rc = ensure_aux(d, count * (size_t)(2 * ctx->nLp));
    if (rc == DKG_OK) rc = launch_pair(ctx, d_bases, d->aux, d_out, d_status, count, stream, mrows, m_limbs);
  } else {
    // aux: inversion area | canonical inverses | pairs.  No host round trip: the redo is predicated
    // on the device-side any_bad, and discards the pair route's results when it runs.
    const size_t inv_words = batchinv_area(ctx, count), plain_words = count * (size_t)ctx->limbs;
    rc = ensure_aux(d, inv_words + plain_words + count * (size_t)(2 * ctx->nLp));
    uint32_t* plain = d->aux + inv_words;
    if (rc == DKG_OK) rc = launch_batchinv(ctx, d_bases, count, plain, stream, &inv);
    if (rc == DKG_OK) rc = launch_pair(ctx, plain, plain + plain_words, d_out, d_status, count, stream, mrows, m_limbs);
    if (rc == DKG_OK) rc = launch_direct(ctx, d_bases, d_out, d_status, nullptr, count, stream, nullptr, inv.any_bad);
  }
  if (rc != DKG_OK || (enc && route != Route::direct)) return rc;
  return launch_range_check(ctx, d_bases, d_out, d_status, count, stream);
}

// shapes for the pair components, in order of preference per padded width
constexpr Shape kNsqShapes[] = {{4, 1}, {4, 2}, {4, 3}, {8, 2}, {6, 3}, {12, 2}, {16, 2}, {12, 3}, {16, 3},
                                {16, 4}, {13, 5}, {14, 5}, {12, 6}, {16, 5}, {16, 6}, {14, 7}, {12, 11}, {16, 9}};

// Constants of the pair arithmetic modulo N (dkg_nsq.cuh, dkg_coop.cuh) for R = 2^(32 L), dense on
// L limbs; a residue c mod N^2 is the pair (c mod N, (c div N) * R mod N).  n, n2: N and N^2.
struct PairConsts {
  dkg_host::Limbs N, ninv, dneg, r2a, r2b, onea, oneb, twoa, twob, plain1, zero;   // ninv: -N^-1 mod 2^(32 K)
  dkg_host::Limbs r2, ninvpos;   // entry / exit: R^2 mod N, N^-1 mod R
};
PairConsts pair_consts(const dkg_host::Limbs& n, const dkg_host::Limbs& n2, int L, int K) {
  using dkg_host::Limbs;
  PairConsts c;
  c.N.assign(L, 0);
  std::copy(n.begin(), n.end(), c.N.begin());
  c.ninv = dkg_host::neg_inv_block(c.N, K);
  c.ninvpos = dkg_host::negate(dkg_host::neg_inv_block(c.N, L));
  const Limbs r = dkg_host::pow2_mod((size_t)32 * L, c.N);
  c.r2 = dkg_host::pow2_mod((size_t)64 * L, c.N);
  c.dneg.assign(L, 0);   // -R mod N
  if (std::any_of(r.begin(), r.end(), [](uint32_t w) { return w != 0; })) { c.dneg = c.N; dkg_host::sub_inplace(c.dneg, r); }
  // pairs of R^2 mod N^2 and R mod N^2: g = g0 + g1 N  ->  (g0, g1 * R mod N)
  auto plain_pair = [&](size_t pow2bits, Limbs* pa, Limbs* pb) {
    Limbs q, g0;
    dkg_host::divmod_slow(dkg_host::pow2_mod(pow2bits, n2), n, &q, &g0);
    pa->assign(L, 0);
    std::copy(g0.begin(), g0.end(), pa->begin());
    Limbs g1(L, 0);
    for (int i = 0; i < (int)q.size() && i < L; ++i) g1[i] = q[i];
    *pb = dkg_host::mulmod_slow(g1, r, c.N);
  };
  plain_pair((size_t)64 * L, &c.r2a, &c.r2b);
  plain_pair((size_t)32 * L, &c.onea, &c.oneb);
  c.plain1.assign(L, 0);
  c.plain1[0] = 1;
  c.zero.assign(L, 0);
  // pair of 2 with 2N added to its a component (Newton step of pair_invert): (2 onea + 2N, 2 oneb - 2R mod N)
  c.twoa.assign(L, 0);
  uint64_t carry = 0;
  for (int i = 0; i < L; ++i) { uint64_t t = (uint64_t)c.onea[i] + c.N[i] + carry; c.twoa[i] = (uint32_t)t; carry = t >> 32; }
  uint32_t c2 = 0;
  for (int i = 0; i < L; ++i) { const uint32_t nc = c.twoa[i] >> 31; c.twoa[i] = (c.twoa[i] << 1) | c2; c2 = nc; }
  c.twob = dkg_host::submod(dkg_host::addmod(c.oneb, c.oneb, c.N), dkg_host::addmod(r, r, c.N), c.N);
  return c;
}

}  // namespace

extern "C" {

int dkg_version(void) { return 100; }

const char* dkg_last_error(void) { return g_err.c_str(); }
}
// error text for the host-only translation units (dkg_wire.cu)
void dkg_set_error(const char* msg) { g_err = msg; }
extern "C" {

int dkg_device_count(int* count) {
  if (!count) return fail(DKG_ERR_INVALID, "null count");
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) { *count = 0; return fail(DKG_ERR_CUDA, cudaGetErrorString(e)); }
  return DKG_OK;
}

unsigned long long dkg_launch_count(void) { return g_launches.load(); }

int dkg_config_set(const char* key, long value) {
  if (!key || value < 0) return fail(DKG_ERR_INVALID, "bad configuration key/value");
  const std::string k(key);
  if (k == "coop_max") { coop_limit(g_coop_max, "DKG_COOP_MAX", kCoopMaxDefault); g_coop_max.store(value); return DKG_OK; }
  if (k == "coop_grouped_max") { g_coop_grouped_max.store(value); return DKG_OK; }
  if (k == "ct_table") { g_ct_table.store(value ? 1 : 0); return DKG_OK; }
  if (k == "time_kernels") { g_time_kernels.store(value ? 1 : 0); return DKG_OK; }
  return fail(DKG_ERR_INVALID, "unknown configuration key");
}
int dkg_config_get(const char* key, long* value) {
  if (!key || !value) return fail(DKG_ERR_INVALID, "null argument");
  const std::string k(key);
  if (k == "coop_max") { *value = (long)coop_limit(g_coop_max, "DKG_COOP_MAX", kCoopMaxDefault); return DKG_OK; }
  if (k == "coop_grouped_max") { *value = (long)coop_limit(g_coop_grouped_max, "DKG_COOP_GROUPED_MAX", kCoopGroupedMaxDefault); return DKG_OK; }
  if (k == "ct_table") { *value = ct_table_setting() ? 1 : 0; return DKG_OK; }
  if (k == "time_kernels") { *value = g_time_kernels.load(); return DKG_OK; }
  return fail(DKG_ERR_INVALID, "unknown configuration key");
}

int dkg_kernel_times(int device, double* ms, int capacity, int* count) {
  if (!count || capacity < 0 || (capacity > 0 && !ms)) return fail(DKG_ERR_INVALID, "null argument");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  std::lock_guard<std::mutex> lk(d->mu);
  CUDA_TRY(cudaSetDevice(d->device));
  int n = 0;
  for (auto& pr : d->ktimes) {
    float t = 0.f;
    if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&t, pr.first, pr.second) == cudaSuccess && n < capacity) ms[n++] = (double)t;
    cudaEventDestroy(pr.first); cudaEventDestroy(pr.second);
  }
  d->ktimes.clear();
  *count = n;
  return DKG_OK;
}

int dkg_modexp_ctx_create(int device, const uint32_t* modulus, int mod_limbs, const uint32_t* exponent,
                          int exp_limbs, int exp_negative, dkg_modexp_ctx** out) {
  if (!modulus || !out || mod_limbs <= 0 || exp_limbs < 0 || (exp_limbs > 0 && !exponent))
    return fail(DKG_ERR_INVALID, "null/empty argument");
  if (mod_limbs > DKG_MAX_LIMBS) return fail(DKG_ERR_UNSUPPORTED, "modulus wider than DKG_MAX_LIMBS");
  if ((modulus[0] & 1u) == 0) return fail(DKG_ERR_INVALID, "modulus must be odd");
  Shape shape;
  if (!pick_shape(mod_limbs, &shape)) return fail(DKG_ERR_UNSUPPORTED, "no kernel shape for this width");
  DeviceState* dev = nullptr;
  int rc = device_state(device, &dev);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));

  auto* ctx = new dkg_modexp_ctx();
  ctx->dev = dev;
  ctx->limbs = mod_limbs;
  ctx->shape = shape;
  ctx->Lp = shape.K * shape.M;
  ctx->negative = exp_negative ? 1 : 0;
  const dkg::ShapeKernels kernels = lookup_kernels(shape.K, shape.M);
  ctx->ct_table = ct_table_setting();
  ctx->kernel = ctx->ct_table ? kernels.fixed_ct : kernels.fixed;
  if (!ctx->kernel) { delete ctx; return fail(DKG_ERR_UNSUPPORTED, "kernel shape not compiled"); }

  const int Lp = ctx->Lp, K = shape.K;
  dkg_host::Limbs n(Lp, 0);
  for (int i = 0; i < mod_limbs; ++i) n[i] = modulus[i];
  dkg_host::Limbs ninv = dkg_host::neg_inv_block(n, K);
  dkg_host::Limbs one_r = dkg_host::pow2_mod((size_t)32 * Lp, n);
  dkg_host::Limbs r2 = dkg_host::pow2_mod((size_t)64 * Lp, n);
  dkg_host::Limbs r3 = dkg_host::pow2_mod((size_t)96 * Lp, n);
  ctx->n0inv = ninv[0];

  std::vector<uint32_t> consts;
  consts.insert(consts.end(), n.begin(), n.end());
  consts.insert(consts.end(), ninv.begin(), ninv.end());
  consts.insert(consts.end(), r2.begin(), r2.end());
  consts.insert(consts.end(), one_r.begin(), one_r.end());
  consts.insert(consts.end(), r3.begin(), r3.end());
  for (const dkg_host::Limbs* v : {&r2, &one_r, &r3}) append_lane_replicated(consts, *v, K);

  // window digits
  ctx->ebits = exp_limbs ? dkg_host::bit_length(exponent, exp_limbs) : 0;
  // Default: fixed windows, every window multiplies (digit 0 by the Montgomery one), so the sequence
  // of operations does not depend on the exponent's bits -- only the table index does.  Sliding
  // windows (DKG_SLIDING_WINDOW=1) save 23 % of the multiplications (~1.5 % of the run time in the
  // pair arithmetic) at the price of an exponent-dependent operation list, as in mpz_powm.
  std::vector<uint32_t> ops;
  if (const char* sw = getenv("DKG_SLIDING_WINDOW"); sw && atoi(sw) != 0 && !ctx->ct_table) {
    ctx->wbits = choose_window(ctx->ebits, 7, sliding_window_cost);
    ops = sliding_window_ops(exponent, ctx->ebits, ctx->wbits, &ctx->tab_entries, &ctx->nmul);
    ctx->table_odd = 1;
  } else {
    ctx->wbits = choose_window(ctx->ebits, 7, ctx->ct_table ? ct_window_cost : fixed_window_cost);
    const int ndigits = (ctx->ebits + ctx->wbits - 1) / ctx->wbits;
    for (int t = 0; t < ndigits; ++t) {
      const int lowbit = ctx->wbits * (ndigits - 1 - t);
      unsigned dgt = 0;
      for (int b = 0; b < ctx->wbits; ++b) {
        const int bit = lowbit + b;
        if (bit < ctx->ebits && ((exponent[bit / 32] >> (bit % 32)) & 1u)) dgt |= 1u << b;
      }
      ops.push_back(((t == 0 ? 0u : (uint32_t)ctx->wbits) << 8) | (dgt ? dgt - 1 : kOpMulOne));
    }
    ctx->tab_entries = ndigits ? (1 << ctx->wbits) - 1 : 0;
    ctx->nmul = ndigits;
    ctx->table_odd = 0;
  }
  ctx->nops = (int)ops.size();
  if (ops.empty()) ops.push_back(0);

  // launch geometry: one CTA per SM, as many warps as shared memory allows (<= 8)
  const size_t uni = (((size_t)(Lp + K) * 4 + 15) / 16) * 16;
  const size_t per_warp = (size_t)Lp * 32 * 4;  // X only: the quotient blocks live in global scratch
  int warps = (int)std::min<size_t>(DKG_MAX_THREADS / 32, (kMaxDynSmem - uni) / per_warp);
  if (warps < 1) { delete ctx; return fail(DKG_ERR_UNSUPPORTED, "operand too wide for shared memory"); }
  ctx->warps = warps;
  ctx->ctas = dev->sm_count;
  ctx->smem = uni + per_warp * warps;
  const size_t tsize = (size_t)ctx->tab_entries + 1;  // odd powers, then the slot of c^2
  // per-warp scratch: window table (also the workspace of the modular inverse: 4 arrays), then Q
  ctx->scratch_q_offset = std::max<size_t>(tsize, 4) * (size_t)Lp * 32;
  ctx->scratch_per_warp = ctx->scratch_q_offset + (size_t)Lp * 32;

  ctx->inv_kernel = kernels.batchinv;
  {
    const size_t inv_per_warp = (size_t)6 * Lp * 32 * 4;
    ctx->inv_warps = (int)std::min<size_t>(2, (kMaxDynSmem - uni) / inv_per_warp);
    if (ctx->inv_warps < 1) ctx->inv_kernel = nullptr;  // too wide: keep the in-kernel inversion
    ctx->inv_smem = uni + inv_per_warp * std::max(ctx->inv_warps, 1);
    if (ctx->inv_kernel) {
      cudaError_t e2 = cudaFuncSetAttribute((const void*)ctx->inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->inv_smem);
      if (e2 != cudaSuccess) { delete ctx; return fail(DKG_ERR_CUDA, std::string("cudaFuncSetAttribute(inv): ") + cudaGetErrorString(e2)); }
    }
  }
  cudaError_t e = cudaFuncSetAttribute((const void*)ctx->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ctx->smem);
  if (e != cudaSuccess) { delete ctx; return fail(DKG_ERR_CUDA, std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e)); }
  e = cudaMalloc(&ctx->d_consts, consts.size() * 4);
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_ops, ops.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(ctx->d_consts, consts.data(), consts.size() * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(ctx->d_ops, ops.data(), ops.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    dkg_modexp_ctx_destroy(ctx);
    return fail(DKG_ERR_CUDA, std::string("context upload: ") + cudaGetErrorString(e));
  }
  *out = ctx;
  return DKG_OK;
}

void dkg_modexp_ctx_destroy(dkg_modexp_ctx* ctx) {
  if (!ctx) return;
  if (ctx->dev) cudaSetDevice(ctx->dev->device);
  if (ctx->d_consts) cudaFree(ctx->d_consts);
  if (ctx->d_ops) cudaFree(ctx->d_ops);
  if (ctx->d_nconsts) cudaFree(ctx->d_nconsts);
  if (ctx->d_nio) cudaFree(ctx->d_nio);
  if (ctx->d_cconsts) cudaFree(ctx->d_cconsts);
  if (ctx->d_cio) cudaFree(ctx->d_cio);
  delete ctx;
}

// Context for the modulus N^2 given its root N: same semantics as dkg_modexp_ctx_create with
// modulus = N*N, but exponentiations run in pair arithmetic modulo N (about 1.6x fewer multiplies).
int dkg_modexp_ctx_create_nsq(int device, const uint32_t* n, int n_limbs, const uint32_t* exponent, int exp_limbs,
                              int exp_negative, dkg_modexp_ctx** out) {
  if (!n || !out || n_limbs <= 0) return fail(DKG_ERR_INVALID, "null/empty argument");
  int ln = n_limbs;
  while (ln > 1 && n[ln - 1] == 0) --ln;
  if ((n[0] & 1u) == 0) return fail(DKG_ERR_INVALID, "modulus must be odd");
  // N^2 and the ordinary context on it (constants for the batched inversion and the fallback)
  const dkg_host::Limbs nn(n, n + ln), n2 = dkg_host::square(nn);
  const int l2 = (int)n2.size();
  dkg_modexp_ctx* ctx = nullptr;
  int rc = dkg_modexp_ctx_create(device, n2.data(), l2, exponent, exp_limbs, exp_negative, &ctx);
  if (rc != DKG_OK) return rc;
  *out = ctx;
  // pair components: R = 2^(32 Lp) >= 8 N
  const int nbits = dkg_host::bit_length(nn.data(), ln);
  if (nbits < 2) return DKG_OK;  // N = 1: nothing to gain
  const int need = (nbits + 3 + 31) / 32;
  Shape sh{};
  dkg::ShapeKernels kernels;
  for (const Shape& c : kNsqShapes)
    if (c.K * c.M >= need && (kernels = lookup_kernels(c.K, c.M)).nsq != nullptr) { sh = c; break; }
  dkg::NsqFn kernel = kernels.nsq;
  if (!kernel || sh.K * sh.M > dkg::kNsqMaxL) return DKG_OK;  // too wide: keep the direct kernel
  // Lp: limbs of the pair components, R = 2^(32 Lp).  In the kernel's memory a block of K limbs
  // occupies a slot of KP = K + (K & 1) limbs (whole 64-bit vectors; odd K: one zero pad limb), a
  // number Ls = KP * M limbs; the entry / exit kernels and the pair rows between them are dense (Lp).
  const int Lp = sh.K * sh.M, K = sh.K, KP = K + (K & 1), Ls = KP * sh.M;
  auto slotted = [&](const dkg_host::Limbs& v) {
    dkg_host::Limbs out((size_t)KP * (v.size() / K), 0);
    for (size_t i = 0; i < v.size(); ++i) out[(i / K) * KP + i % K] = v[i];
    return out;
  };
  const PairConsts pc = pair_consts(nn, n2, Lp, K);
  std::vector<uint32_t> kc;
  for (const dkg_host::Limbs* v : {&pc.N, &pc.ninv, &pc.dneg, &pc.r2a, &pc.r2b, &pc.onea, &pc.oneb, &pc.plain1, &pc.zero}) {
    const dkg_host::Limbs sv = slotted(*v);
    kc.insert(kc.end(), sv.begin(), sv.end());
  }
  for (const dkg_host::Limbs* v : {&pc.r2a, &pc.r2b, &pc.onea, &pc.oneb, &pc.plain1, &pc.zero}) append_lane_replicated(kc, slotted(*v), KP);
  for (const dkg_host::Limbs* v : {&pc.twoa, &pc.twob}) {
    const dkg_host::Limbs sv = slotted(*v);
    kc.insert(kc.end(), sv.begin(), sv.end());
  }
  std::vector<uint32_t> ioc;
  for (const dkg_host::Limbs* v : {&pc.N, &pc.r2, &pc.ninvpos}) ioc.insert(ioc.end(), v->begin(), v->end());

  const size_t uni = (((size_t)(2 * Ls + KP + Lp) * 4 + 15) / 16) * 16 +
                     (((size_t)dkg::sched_total_words_closed(sh.M) * 4 + 15) / 16) * 16;  // consts | schedule table
  size_t per_warp = (size_t)2 * Ls * 32 * 4;
  int maxw = DKG_MAX_THREADS / 32;
  int warps = (int)std::min<size_t>(maxw, (kMaxDynSmem - uni) / per_warp);
  // wide keys: shared memory, not registers, caps the warps per SM; with fewer than 10 take the
  // variant that keeps the b component in global scratch (a only in shared memory)
  bool bg = false;
  if (warps < 10 && env_long("DKG_NSQ_BG", 1) != 0 && kernels.nsq_bg != nullptr) {
    kernel = kernels.nsq_bg; bg = true;
    per_warp = (size_t)Ls * 32 * 4;
    warps = (int)std::min<size_t>(maxw, (kMaxDynSmem - uni) / per_warp);
  }
  if (warps < 1) return DKG_OK;
  // window table (odd powers, then the slot of c^2 / the constant-time spare), then 4 pair slots of
  // work space for the in-kernel inversion of negative exponents
  const size_t tsize = (size_t)ctx->tab_entries + 1;
  ctx->ninv_slot = std::max<size_t>(tsize, 1);
  // (off by default: measured 0.5 % slower than the batched inversion kernel, whose one GCD per chain
  // runs beside idle SMs, while these GCDs -- one per ciphertext, divergent -- take the exponentiation
  // kernel's own time; what it buys is an exact per-element status without the predicated redo)
  ctx->nsq_inv = env_long("DKG_INKERNEL_INVERSE", 0) != 0;
  ctx->nscratch_q_offset = (ctx->ninv_slot + 4) * 2 * (size_t)Ls * 32;
  ctx->nscratch_per_warp = ctx->nscratch_q_offset + (size_t)Ls * 32 * (bg ? 2 : 1);   // Q [| b]
  ctx->nsq_bg = bg;
  cudaError_t e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(uni + per_warp * warps));
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_nconsts, kc.size() * 4);
  if (e == cudaSuccess) e = cudaMalloc(&ctx->d_nio, ioc.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(ctx->d_nconsts, kc.data(), kc.size() * 4, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(ctx->d_nio, ioc.data(), ioc.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) {
    dkg_modexp_ctx_destroy(ctx);
    *out = nullptr;
    return fail(DKG_ERR_CUDA, std::string("nsq context: ") + cudaGetErrorString(e));
  }
  ctx->nshape = sh; ctx->nLp = Lp; ctx->nLs = Ls; ctx->nwarps = warps; ctx->nsmem = uni + per_warp * warps;
  ctx->n_n0inv = pc.ninv[0]; ctx->nsq_kernel = kernel; ctx->nsq = true;

  // ---- cooperative (warp-per-operand) latency path, dkg_coop.cuh: its own R = 2^(32 cLc) >= 8N -----
  int cK = 0, cnb = 0;
  const size_t coop_max = coop_limit(g_coop_max, "DKG_COOP_MAX", kCoopMaxDefault);
  if (coop_max > 0 && coop_shape(need, &cK, &cnb) && cK * cnb <= dkg::kNsqMaxL) {
    const int Lc = cK * cnb;
    const PairConsts cp = pair_consts(nn, n2, Lc, Lc);
    std::vector<uint32_t> cc, cio;
    for (const dkg_host::Limbs* v : {&cp.N, &cp.ninv, &cp.dneg, &cp.r2a, &cp.r2b, &cp.onea, &cp.oneb, &cp.twoa, &cp.twob, &cp.plain1, &cp.zero})
      cc.insert(cc.end(), v->begin(), v->end());
    for (const dkg_host::Limbs* v : {&cp.N, &cp.r2, &cp.ninvpos}) cio.insert(cio.end(), v->begin(), v->end());
    cudaError_t e2 = cudaMalloc(&ctx->d_cconsts, cc.size() * 4);
    if (e2 == cudaSuccess) e2 = cudaMalloc(&ctx->d_cio, cio.size() * 4);
    if (e2 == cudaSuccess) e2 = cudaMemcpy(ctx->d_cconsts, cc.data(), cc.size() * 4, cudaMemcpyHostToDevice);
    if (e2 == cudaSuccess) e2 = cudaMemcpy(ctx->d_cio, cio.data(), cio.size() * 4, cudaMemcpyHostToDevice);
    if (e2 != cudaSuccess) {
      dkg_modexp_ctx_destroy(ctx);
      *out = nullptr;
      return fail(DKG_ERR_CUDA, std::string("cooperative-path constants: ") + cudaGetErrorString(e2));
    }
    ctx->cK = cK; ctx->cnb = cnb; ctx->cLc = Lc; ctx->coop_max = coop_max;
    ctx->cfull = make_coop_plan(cnb, 2 * cnb - 1);
    ctx->clow = make_coop_plan(cnb, cnb);
    ctx->coop = true;
  }
  return DKG_OK;
}

int dkg_modexp_ctx_info(const dkg_modexp_ctx* ctx, int info[12]) {
  if (!ctx || !info) return fail(DKG_ERR_INVALID, "null argument");
  info[0] = ctx->shape.K; info[1] = ctx->shape.M; info[2] = ctx->Lp; info[3] = ctx->wbits;
  info[4] = ctx->nmul; info[5] = ctx->ebits; info[6] = ctx->warps; info[7] = ctx->ctas;
  info[8] = ctx->nsq ? 1 : 0; info[9] = ctx->nshape.K; info[10] = ctx->nshape.M; info[11] = ctx->nwarps;
  return DKG_OK;
}

int dkg_modexp_batch_device(dkg_modexp_ctx* ctx, const uint32_t* d_bases, uint32_t* d_out,
                            uint8_t* d_status, size_t count, void* stream) {
  if (!ctx || (count && (!d_bases || !d_out))) return fail(DKG_ERR_INVALID, "null argument");
  DeviceLease lease(ctx->dev, (cudaStream_t)stream);
  return launch_modexp(ctx, d_bases, d_out, d_status, count, (cudaStream_t)stream);
}

int dkg_modexp_batch(dkg_modexp_ctx* ctx, const uint32_t* bases, uint32_t* out, uint8_t* status,
                     size_t count) {
  if (!ctx || (count && (!bases || !out))) return fail(DKG_ERR_INVALID, "null argument");
  if (count == 0) return DKG_OK;
  DeviceState* d = ctx->dev;
  CUDA_TRY(cudaSetDevice(d->device));
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  const size_t bytes = count * (size_t)ctx->limbs * 4;
  uint32_t *d_in, *d_out;
  uint8_t* d_st;
  cudaError_t e = bufs.alloc(&d_in, bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_out, bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_st, count);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("batch alloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_in, bases, bytes, cudaMemcpyHostToDevice, d->stream));
  int rc = launch_modexp(ctx, d_in, d_out, d_st, count, d->stream);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, bytes, cudaMemcpyDeviceToHost, d->stream));
  if (status) CUDA_TRY(cudaMemcpyAsync(status, d_st, count, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

}  // extern "C"

// ---- share combination ---------------------------------------------------------------------------
struct dkg_combine_ctx {
  DeviceState* dev = nullptr;
  int ln = 0, l2 = 0, shares = 0;
  uint32_t n2_0inv = 0, n_0inv = 0;
  uint32_t* d_consts = nullptr;
  // warp-per-ciphertext kernel (dkg_coop.cuh: coop_combine_kernel), used whenever N^2 fits its shapes
  bool coop = false;
  int cK = 0, cnb = 0;
  uint32_t* d_cconsts = nullptr;
  dkg::CoopPlanTable cfull{}, clow{};
};

namespace {
int launch_combine(dkg_combine_ctx* ctx, const uint32_t* d_partials, uint32_t* d_out, uint8_t* d_status,
                   size_t count, cudaStream_t stream) {
  if (count == 0) return DKG_OK;
  CUDA_TRY(cudaSetDevice(ctx->dev->device));
  if (ctx->coop) {
    DeviceState* d = ctx->dev;
    const int Lc = ctx->cK * ctx->cnb;
    int ctas = 1, warps = 1;
    coop_grid(d, ctx->cK, ctx->cK == 12, count, &ctas, &warps);
    CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), stream));
    dkg::CoopCombineParams q{};
    q.partials = d_partials; q.out = d_out; q.status = d_status; q.count = count; q.shares = ctx->shares; q.l2 = ctx->l2;
    q.ln = ctx->ln; q.nb = ctx->cnb; q.consts = ctx->d_cconsts; q.counter = d->counter; q.full = ctx->cfull; q.low = ctx->clow;
    const size_t smem = ((size_t)dkg::kCoopCombineConsts + (size_t)dkg::kCoopCombineWarpBufs * warps) * Lc * 4;
    CUDA_TRY(dkg::launch_coop_combine(ctx->cK, q, ctas, warps, smem, stream));
    g_launches.fetch_add(1);
    return DKG_OK;
  }
  dkg::CombineParams p{};
  p.partials = d_partials; p.out = d_out; p.status = d_status; p.count = count; p.shares = ctx->shares;
  p.l2 = ctx->l2; p.ln = ctx->ln; p.consts = ctx->d_consts; p.n2_0inv = ctx->n2_0inv; p.n_0inv = ctx->n_0inv;
  const int threads = 128;
  const unsigned blocks = (unsigned)((count + threads - 1) / threads);
  dkg::combine_kernel<<<blocks, threads, 0, stream>>>(p);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(1);
  return DKG_OK;
}
}  // namespace

extern "C" {

int dkg_combine_ctx_create(int device, const uint32_t* n, int n_limbs, const uint32_t* theta_inv, int shares,
                           dkg_combine_ctx** out) {
  if (!n || !theta_inv || !out || n_limbs <= 0 || shares < 1) return fail(DKG_ERR_INVALID, "null/empty argument");
  if ((n[0] & 1u) == 0) return fail(DKG_ERR_INVALID, "modulus must be odd");
  int ln = n_limbs;
  while (ln > 1 && n[ln - 1] == 0) --ln;
  if (ln > dkg::kCombineMaxL - 1) return fail(DKG_ERR_UNSUPPORTED, "N wider than the combine kernel supports");
  DeviceState* dev = nullptr;
  int rc = device_state(device, &dev);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  const dkg_host::Limbs nn(n, n + ln), n2 = dkg_host::square(nn);
  const int l2 = (int)n2.size();
  dkg_host::Limbs rpow = dkg_host::pow2_mod((size_t)32 * l2 * shares, n2);
  dkg_host::Limbs ninvneg = dkg_host::neg_inv_block(nn, ln);
  dkg_host::Limbs ninvpos = dkg_host::negate(ninvneg);
  dkg_host::Limbs th(ln, 0);
  for (int i = 0; i < ln && i < n_limbs; ++i) th[i] = theta_inv[i];
  if (!dkg_host::geq(nn, th) || th == nn) return fail(DKG_ERR_INVALID, "theta_inv must be < N");
  dkg_host::Limbs thr = dkg_host::mulmod_slow(th, dkg_host::pow2_mod((size_t)32 * ln, nn), nn);

  auto* ctx = new dkg_combine_ctx();
  ctx->dev = dev; ctx->ln = ln; ctx->l2 = l2; ctx->shares = shares;
  ctx->n2_0inv = dkg_host::neg_inv_block(n2, 1)[0];
  ctx->n_0inv = ninvneg[0];
  std::vector<uint32_t> consts;
  consts.insert(consts.end(), n2.begin(), n2.end());
  consts.insert(consts.end(), rpow.begin(), rpow.end());
  consts.insert(consts.end(), nn.begin(), nn.end());
  consts.insert(consts.end(), ninvpos.begin(), ninvpos.end());
  consts.insert(consts.end(), thr.begin(), thr.end());
  cudaError_t e = cudaMalloc(&ctx->d_consts, consts.size() * 4);
  if (e == cudaSuccess) e = cudaMemcpy(ctx->d_consts, consts.data(), consts.size() * 4, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { dkg_combine_ctx_destroy(ctx); return fail(DKG_ERR_CUDA, std::string("combine ctx: ") + cudaGetErrorString(e)); }
  // warp-per-ciphertext kernel: R = 2^(32 Lc) >= 4 N^2
  {
    const int n2bits = dkg_host::bit_length(n2.data(), l2);
    int cK = 0, cnb = 0;
    if (env_long("DKG_COOP_COMBINE", 1) != 0 && coop_shape((n2bits + 2 + 31) / 32, &cK, &cnb)) {
      const int Lc = cK * cnb;
      dkg_host::Limbs N2c(Lc, 0), Nc(Lc, 0), thc(Lc, 0);
      for (int i = 0; i < l2; ++i) N2c[i] = n2[i];
      for (int i = 0; i < ln; ++i) { Nc[i] = nn[i]; thc[i] = th[i]; }
      dkg_host::Limbs ni2 = dkg_host::neg_inv_block(N2c, Lc), nin = dkg_host::neg_inv_block(Nc, Lc);
      dkg_host::Limbs rpow_c = dkg_host::pow2_mod((size_t)32 * Lc * shares, N2c);
      dkg_host::Limbs thr_c = dkg_host::mulmod_slow(thc, dkg_host::pow2_mod((size_t)32 * Lc, Nc), Nc);
      std::vector<uint32_t> cc;
      for (const dkg_host::Limbs* v : {&N2c, &ni2, &rpow_c, &Nc, &nin, &thr_c}) cc.insert(cc.end(), v->begin(), v->end());
      cudaError_t e2 = cudaMalloc(&ctx->d_cconsts, cc.size() * 4);
      if (e2 == cudaSuccess) e2 = cudaMemcpy(ctx->d_cconsts, cc.data(), cc.size() * 4, cudaMemcpyHostToDevice);
      if (e2 != cudaSuccess) { dkg_combine_ctx_destroy(ctx); return fail(DKG_ERR_CUDA, std::string("combine ctx (cooperative constants): ") + cudaGetErrorString(e2)); }
      ctx->cK = cK; ctx->cnb = cnb;
      ctx->cfull = make_coop_plan(cnb, 2 * cnb - 1);
      ctx->clow = make_coop_plan(cnb, cnb);
      ctx->coop = true;
    }
  }
  *out = ctx;
  return DKG_OK;
}

void dkg_combine_ctx_destroy(dkg_combine_ctx* ctx) {
  if (!ctx) return;
  if (ctx->dev) cudaSetDevice(ctx->dev->device);
  if (ctx->d_consts) cudaFree(ctx->d_consts);
  if (ctx->d_cconsts) cudaFree(ctx->d_cconsts);
  delete ctx;
}

int dkg_combine_n2_limbs(const dkg_combine_ctx* ctx) { return ctx ? ctx->l2 : 0; }

int dkg_combine_batch_device(dkg_combine_ctx* ctx, const uint32_t* d_partials, uint32_t* d_out, uint8_t* d_status,
                             size_t count, void* stream) {
  if (!ctx || (count && (!d_partials || !d_out))) return fail(DKG_ERR_INVALID, "null argument");
  DeviceLease lease(ctx->dev, (cudaStream_t)stream);
  return launch_combine(ctx, d_partials, d_out, d_status, count, (cudaStream_t)stream);
}

int dkg_combine_batch(dkg_combine_ctx* ctx, const uint32_t* partials, uint32_t* out, uint8_t* status, size_t count) {
  if (!ctx || (count && (!partials || !out))) return fail(DKG_ERR_INVALID, "null argument");
  if (count == 0) return DKG_OK;
  DeviceState* d = ctx->dev;
  CUDA_TRY(cudaSetDevice(d->device));
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  const size_t in_bytes = (size_t)ctx->shares * count * ctx->l2 * 4, out_bytes = count * (size_t)ctx->ln * 4;
  uint32_t *d_in, *d_out;
  uint8_t* d_st;
  cudaError_t e = bufs.alloc(&d_in, in_bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_out, out_bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_st, count);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("combine alloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_in, partials, in_bytes, cudaMemcpyHostToDevice, d->stream));
  int rc = launch_combine(ctx, d_in, d_out, d_st, count, d->stream);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, d->stream));
  if (status) CUDA_TRY(cudaMemcpyAsync(status, d_st, count, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

}  // extern "C"

// ---- encryption: (1 + m N) * r^N mod N^2 ----------------------------------------------------------
extern "C" int dkg_encrypt_batch(dkg_modexp_ctx* ctx, const uint32_t* n, int n_limbs, const uint32_t* r,
                                 const uint32_t* m, uint32_t* out, size_t count) {
  if (!ctx || !n || n_limbs <= 0 || (count && (!r || !out))) return fail(DKG_ERR_INVALID, "null argument");
  if (n_limbs > ctx->limbs) return fail(DKG_ERR_INVALID, "n wider than the context modulus");
  if (ctx->negative) return fail(DKG_ERR_INVALID, "encryption needs a context with a positive exponent (N)");
  if (count == 0) return DKG_OK;
  DeviceState* d = ctx->dev;
  CUDA_TRY(cudaSetDevice(d->device));
  const size_t in_bytes = count * (size_t)n_limbs * 4, out_bytes = count * (size_t)ctx->limbs * 4;
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_r, *d_m = nullptr, *d_n, *d_base, *d_fm = nullptr, *d_out;
  cudaError_t e = bufs.alloc(&d_r, in_bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_base, out_bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_out, out_bytes);
  if (e == cudaSuccess) e = bufs.alloc(&d_n, (size_t)n_limbs * 4);
  if (e == cudaSuccess && m) e = bufs.alloc(&d_m, in_bytes);
  if (e == cudaSuccess && m) e = bufs.alloc(&d_fm, out_bytes);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("encrypt alloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_r, r, in_bytes, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_n, n, (size_t)n_limbs * 4, cudaMemcpyHostToDevice, d->stream));
  if (m) CUDA_TRY(cudaMemcpyAsync(d_m, m, in_bytes, cudaMemcpyHostToDevice, d->stream));
  const unsigned blocks = (unsigned)std::min<size_t>((count * ctx->limbs + 255) / 256, 148 * 16);
  dkg::pad_rows_kernel<<<blocks, 256, 0, d->stream>>>(d_r, n_limbs, d_base, ctx->limbs, count);
  g_launches.fetch_add(1);
  if (m) {
    dkg::one_plus_mn_kernel<<<(unsigned)((count + 127) / 128), 128, 0, d->stream>>>(d_m, d_n, n_limbs, d_fm, ctx->limbs, count);
    g_launches.fetch_add(1);
  }
  CUDA_TRY(cudaGetLastError());
  const EncryptFactor enc{d_m, n_limbs, d_fm};
  int rc = launch_modexp(ctx, d_base, d_out, nullptr, count, d->stream, &enc);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

// ---- grouped modexp (biprimality test batch) -------------------------------------------------------
namespace {

struct GroupedPlan {
  Shape shape{};
  dkg::GroupedFn kernel = nullptr;
  int Lp = 0, K = 0, Ka = 0, wbits = 1, ndigits = 1, warps = 1, ctas = 1;   // K, Lp: slot layout; Ka: arithmetic block
  size_t smem = 0, q_off = 0, scratch_per_warp = 0;
  bool ct_table = false;   // constant-time table access: narrower windows, one more table slot
};

int plan_grouped(DeviceState* d, int limbs, int ebits, size_t count, bool ct_table, GroupedPlan* plan) {
  if (const char* f = getenv("DKG_GROUPED_SHAPE")) {  // tuning knob: "K,M"
    int k = 0, m = 0;
    if (sscanf(f, "%d,%d", &k, &m) == 2 && k * m >= limbs && (plan->kernel = lookup_kernels(k, m).grouped) != nullptr) plan->shape = Shape{k, m};
  }
  // by padded width, except that K = 22 (spills at 168 registers) yields to (14,5): measured
  // 304 k vs 222 k modexps/s on 65-limb candidates
  static constexpr Shape kGroupedPref[] = {
      {4, 1}, {4, 2}, {4, 3}, {8, 2}, {6, 3}, {12, 2}, {16, 2}, {12, 3}, {16, 3}, {16, 4},
      {13, 5}, {14, 5}, {22, 3}, {16, 5}, {16, 6}, {16, 8}, {12, 11},
  };
  if (!plan->kernel)
    for (const Shape& sh : kGroupedPref)
      if (sh.K * sh.M >= limbs && (plan->kernel = lookup_kernels(sh.K, sh.M).grouped) != nullptr) { plan->shape = sh; break; }
  if (!plan->kernel)
    for (const Shape& sh : kShapes)
      if (sh.K * sh.M >= limbs && (plan->kernel = lookup_kernels(sh.K, sh.M).grouped) != nullptr) { plan->shape = sh; break; }
  if (!plan->kernel) return fail(DKG_ERR_UNSUPPORTED, "modulus wider than the grouped kernel shapes (132 limbs)");
  plan->Ka = plan->shape.K;
  plan->K = plan->shape.K + (plan->shape.K & 1);
  plan->Lp = plan->K * plan->shape.M;
  plan->ct_table = ct_table;
  if (ct_table) plan->kernel = lookup_kernels(plan->shape.K, plan->shape.M).grouped_ct;   // (compiled with .grouped)
  plan->wbits = choose_window(ebits, 6, ct_table ? ct_window_cost : fixed_window_cost);
  plan->ndigits = std::max(1, (ebits + plan->wbits - 1) / plan->wbits);
  const size_t per_warp_smem = ((size_t)2 * plan->Lp + plan->K) * 32 * 4;
  const size_t sched_bytes = (((size_t)dkg::sched_total_words_closed(plan->shape.M) * 4 + 15) / 16) * 16;
  plan->warps = (int)std::min<size_t>(DKG_MAX_THREADS / 32, (kMaxDynSmem - sched_bytes) / per_warp_smem);
  if (plan->warps < 1) return fail(DKG_ERR_UNSUPPORTED, "operand too wide for shared memory");
  plan->smem = sched_bytes + per_warp_smem * plan->warps;
  const size_t tsize = ((size_t)1 << plan->wbits) - 1 + (ct_table ? 1 : 0);   // (+ the slot ct_select writes)
  plan->q_off = std::max<size_t>(tsize, 1) * (size_t)plan->Lp * 32;
  plan->scratch_per_warp = plan->q_off + (size_t)3 * plan->Lp * 32;  // Q | R2 | ONER in lane layout
  plan->ctas = wave_ctas(d->sm_count, plan->warps, count);
  int rc = ensure_scratch(d, (size_t)d->sm_count * plan->warps * plan->scratch_per_warp);
  if (rc != DKG_OK) return rc;
  cudaError_t e = cudaFuncSetAttribute((const void*)plan->kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan->smem);
  if (e != cudaSuccess) return fail(DKG_ERR_CUDA, std::string("cudaFuncSetAttribute(grouped): ") + cudaGetErrorString(e));
  return DKG_OK;
}

// Cooperative (warp-per-operand) variant for small candidate batches, dkg_coop.cuh: needs no
// per-group constants (each warp derives -N^-1, R, R^2 for its instance) and no setup kernel.
struct CoopGroupedPlan {
  int K = 0, nb = 0, Lc = 0, wbits = 1, ndigits = 1, ctas = 1, warps = 1;
  size_t smem = 0, per_warp = 0;
  dkg::CoopPlanTable full{}, low{};
  bool ct_table = false;   // constant-time table access (the selection goes to Y: no extra slot)
};

// true if this batch should take the cooperative kernel (moduli: host copy, for the widest one)
bool plan_coop_grouped(DeviceState* d, const uint32_t* moduli, size_t groups, int limbs, int ebits, size_t count,
                       bool ct_table, CoopGroupedPlan* plan) {
  if (count == 0 || count > coop_limit(g_coop_grouped_max, "DKG_COOP_GROUPED_MAX", kCoopGroupedMaxDefault)) return false;
  int maxbits = 1;
  for (size_t g = 0; g < groups; ++g) maxbits = std::max(maxbits, dkg_host::bit_length(moduli + g * (size_t)limbs, limbs));
  const int need = (maxbits + 2 + 31) / 32;   // R >= 4N
  if (!coop_shape(need, &plan->K, &plan->nb)) return false;
  plan->Lc = plan->K * plan->nb;
  plan->ct_table = ct_table;
  plan->wbits = choose_window(ebits, 6, ct_table ? ct_window_cost : fixed_window_cost);
  plan->ndigits = std::max(1, (ebits + plan->wbits - 1) / plan->wbits);
  coop_grid(d, plan->K, false, count, &plan->ctas, &plan->warps);
  plan->smem = (size_t)9 * plan->warps * plan->Lc * 4;
  plan->per_warp = (((size_t)1 << plan->wbits) - 1) * plan->Lc;
  plan->full = make_coop_plan(plan->nb, 2 * plan->nb - 1);
  plan->low = make_coop_plan(plan->nb, plan->nb);
  return true;
}

int launch_coop_grouped_batch(DeviceState* d, const CoopGroupedPlan& plan, const uint32_t* d_mod, const uint32_t* d_exp,
                              int exp_limbs, const uint32_t* d_bases, uint32_t* d_out, size_t groups, int per_group, int limbs) {
  int rc = ensure_scratch(d, (size_t)plan.ctas * plan.warps * plan.per_warp);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), d->stream));
  dkg::CoopGroupedParams p{};
  p.moduli = d_mod; p.exps = d_exp; p.bases = d_bases; p.out = d_out; p.groups = groups; p.per_group = per_group;
  p.limbs = limbs; p.exp_limbs = exp_limbs; p.nb = plan.nb; p.wbits = plan.wbits; p.ndigits = plan.ndigits;
  p.scratch = d->scratch; p.scratch_per_warp = plan.per_warp; p.counter = d->counter; p.full = plan.full; p.low = plan.low;
  CUDA_TRY(dkg::launch_coop_grouped(plan.K, plan.ct_table, p, plan.ctas, plan.warps, plan.smem, d->stream));
  g_launches.fetch_add(1);
  return DKG_OK;
}

// Grouped modexp of groups x per_group device rows on d->stream: the cooperative kernel for small
// batches, else group setup + wave kernel with per-group constants and digits allocated in `bufs`.
// moduli, exps: host copies (the plans size themselves for the widest modulus and exponent).
// The constant-time setting ("ct_table") is read on every call.
int launch_grouped(DeviceState* d, DevBufs& bufs, const uint32_t* moduli, const uint32_t* exps, const uint32_t* d_mod,
                   const uint32_t* d_exp, int exp_limbs, const uint32_t* d_bases, uint32_t* d_out, size_t groups,
                   int per_group, int limbs) {
  int ebits = 0;
  for (size_t g = 0; g < groups; ++g) ebits = std::max(ebits, dkg_host::bit_length(exps + g * (size_t)exp_limbs, exp_limbs));
  const size_t count = groups * (size_t)per_group;
  const bool ct_table = ct_table_setting();
  CoopGroupedPlan cplan;
  if (plan_coop_grouped(d, moduli, groups, limbs, ebits, count, ct_table, &cplan))
    return launch_coop_grouped_batch(d, cplan, d_mod, d_exp, exp_limbs, d_bases, d_out, groups, per_group, limbs);
  GroupedPlan plan;
  int rc = plan_grouped(d, limbs, ebits, count, ct_table, &plan);
  if (rc != DKG_OK) return rc;
  uint32_t* d_gc;
  uint8_t* d_dig;
  cudaError_t e = bufs.alloc(&d_gc, groups * (size_t)(3 * plan.Lp + plan.K) * 4);
  if (e == cudaSuccess) e = bufs.alloc(&d_dig, groups * (size_t)plan.ndigits);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("grouped cudaMalloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), d->stream));
  dkg::GroupedParams p{};
  p.moduli = d_mod; p.exps = d_exp; p.bases = d_bases; p.out = d_out; p.groups = groups;
  p.per_group = per_group; p.limbs = limbs; p.exp_limbs = exp_limbs; p.K = plan.K; p.Lp = plan.Lp; p.Ka = plan.Ka;
  p.wbits = plan.wbits; p.ndigits = plan.ndigits; p.gconsts = d_gc; p.digits = d_dig; p.scratch = d->scratch;
  p.scratch_per_warp = plan.scratch_per_warp; p.scratch_q_offset = plan.q_off; p.counter = d->counter;
  dkg::launch_group_setup(p, plan.ct_table, d->stream);
  plan.kernel<<<plan.ctas, plan.warps * 32, plan.smem, d->stream>>>(p);
  g_launches.fetch_add(2);
  CUDA_TRY(cudaGetLastError());
  return DKG_OK;
}


}  // namespace

extern "C" int dkg_modexp_grouped(int device, const uint32_t* moduli, const uint32_t* exps, int exp_limbs,
                                  const uint32_t* bases, uint32_t* out, size_t groups, int per_group, int limbs) {
  if (!moduli || !exps || !bases || !out || exp_limbs <= 0 || per_group <= 0 || limbs <= 0)
    return fail(DKG_ERR_INVALID, "null/empty argument");
  if (groups == 0) return DKG_OK;
  for (size_t g = 0; g < groups; ++g)
    if ((moduli[g * (size_t)limbs] & 1u) == 0) return fail(DKG_ERR_INVALID, "every modulus must be odd");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  const size_t count = groups * (size_t)per_group;
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_mod, *d_exp, *d_bases, *d_out;
  const size_t mod_b = groups * (size_t)limbs * 4, exp_b = groups * (size_t)exp_limbs * 4, base_b = count * (size_t)limbs * 4;
  cudaError_t e = bufs.alloc(&d_mod, mod_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_exp, exp_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_bases, base_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_out, base_b);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("grouped cudaMalloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_mod, moduli, mod_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_exp, exps, exp_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_bases, bases, base_b, cudaMemcpyHostToDevice, d->stream));
  rc = launch_grouped(d, bufs, moduli, exps, d_mod, d_exp, exp_limbs, d_bases, d_out, groups, per_group, limbs);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, d_out, base_b, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

// Whole v calculation of one compute_modulus round: Jacobi filter, selection of the first
// `correct` usable g's per candidate, grouped modexp.
extern "C" int dkg_biprime_v_batch(int device, const uint32_t* moduli, const uint32_t* exps, int exp_limbs,
                                   const uint32_t* gvals, int g_per_candidate, int correct, uint32_t* out_v,
                                   int32_t* out_count, size_t groups, int limbs) {
  if (!moduli || !exps || !gvals || !out_v || !out_count || exp_limbs <= 0 || g_per_candidate <= 0 || correct <= 0 || limbs <= 0)
    return fail(DKG_ERR_INVALID, "null/empty argument");
  if (limbs > dkg::kGroupedMaxLimbs) return fail(DKG_ERR_UNSUPPORTED, "candidate wider than the biprime kernels support");
  if (groups == 0) return DKG_OK;
  for (size_t g = 0; g < groups; ++g)
    if ((moduli[g * (size_t)limbs] & 1u) == 0) return fail(DKG_ERR_INVALID, "every modulus must be odd");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  const size_t count = groups * (size_t)correct;
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_mod, *d_exp, *d_g, *d_bases, *d_out;
  int8_t* d_sym;
  int *d_pick, *d_count;
  const size_t mod_b = groups * (size_t)limbs * 4, exp_b = groups * (size_t)exp_limbs * 4;
  const size_t g_b = groups * (size_t)g_per_candidate * limbs * 4, base_b = count * (size_t)limbs * 4;
  cudaError_t e = bufs.alloc(&d_mod, mod_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_exp, exp_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_g, g_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_bases, base_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_out, base_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_sym, groups * (size_t)g_per_candidate);
  if (e == cudaSuccess) e = bufs.alloc(&d_pick, count * sizeof(int));
  if (e == cudaSuccess) e = bufs.alloc(&d_count, groups * sizeof(int));
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("biprime cudaMalloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_mod, moduli, mod_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_exp, exps, exp_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_g, gvals, g_b, cudaMemcpyHostToDevice, d->stream));
  const unsigned long long nsym = groups * (unsigned long long)g_per_candidate;
  dkg::jacobi_kernel<<<(unsigned)((nsym + 127) / 128), 128, 0, d->stream>>>(d_mod, d_g, limbs, groups, g_per_candidate, d_sym);
  dkg::select_g_kernel<<<(unsigned)((groups + 127) / 128), 128, 0, d->stream>>>(d_sym, groups, g_per_candidate, correct, d_pick, d_count);
  const unsigned gblocks = (unsigned)std::min<size_t>((count * limbs + 255) / 256, 148 * 32);
  dkg::gather_g_kernel<<<gblocks, 256, 0, d->stream>>>(d_g, d_pick, limbs, groups, g_per_candidate, correct, d_bases);
  g_launches.fetch_add(3);
  CUDA_TRY(cudaGetLastError());
  rc = launch_grouped(d, bufs, moduli, exps, d_mod, d_exp, exp_limbs, d_bases, d_out, groups, correct, limbs);
  if (rc != DKG_OK) return rc;
  dkg::clear_unused_kernel<<<gblocks, 256, 0, d->stream>>>(d_out, d_count, limbs, groups, correct);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(out_v, d_out, base_b, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaMemcpyAsync(out_count, d_count, groups * sizeof(int), cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

// Jacobi symbols only: sym[g][k] = (gvals[g][k] / moduli[g]) in {-1, 0, 1}
extern "C" int dkg_jacobi_batch(int device, const uint32_t* moduli, const uint32_t* gvals, int per_group, int8_t* sym,
                                size_t groups, int limbs) {
  if (!moduli || !gvals || !sym || per_group <= 0 || limbs <= 0) return fail(DKG_ERR_INVALID, "null/empty argument");
  if (limbs > dkg::kGroupedMaxLimbs) return fail(DKG_ERR_UNSUPPORTED, "operand wider than the Jacobi kernel supports");
  if (groups == 0) return DKG_OK;
  for (size_t g = 0; g < groups; ++g)
    if ((moduli[g * (size_t)limbs] & 1u) == 0) return fail(DKG_ERR_INVALID, "every modulus must be odd");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_mod, *d_g;
  int8_t* d_sym;
  const size_t mod_b = groups * (size_t)limbs * 4, g_b = groups * (size_t)per_group * limbs * 4;
  cudaError_t e = bufs.alloc(&d_mod, mod_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_g, g_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_sym, groups * (size_t)per_group);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("jacobi cudaMalloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_mod, moduli, mod_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_g, gvals, g_b, cudaMemcpyHostToDevice, d->stream));
  const unsigned long long nsym = groups * (unsigned long long)per_group;
  dkg::jacobi_kernel<<<(unsigned)((nsym + 127) / 128), 128, 0, d->stream>>>(d_mod, d_g, limbs, groups, per_group, d_sym);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(sym, d_sym, groups * (size_t)per_group, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

// flags[g] = 1 if moduli[g] has a divisor among primes[0..nprimes)
extern "C" int dkg_small_prime_sieve(int device, const uint32_t* moduli, const uint32_t* primes, int nprimes,
                                     uint8_t* flags, size_t groups, int limbs) {
  if (!moduli || !primes || !flags || nprimes <= 0 || limbs <= 0) return fail(DKG_ERR_INVALID, "null/empty argument");
  if (groups == 0) return DKG_OK;
  for (int k = 0; k < nprimes; ++k)
    if (primes[k] < 2) return fail(DKG_ERR_INVALID, "primes must be >= 2");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_mod, *d_pr;
  uint8_t* d_fl;
  const size_t mod_b = groups * (size_t)limbs * 4;
  cudaError_t e = bufs.alloc(&d_mod, mod_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_pr, (size_t)nprimes * 4);
  if (e == cudaSuccess) e = bufs.alloc(&d_fl, groups);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("sieve cudaMalloc: ") + cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(d_mod, moduli, mod_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_pr, primes, (size_t)nprimes * 4, cudaMemcpyHostToDevice, d->stream));
  for (size_t off = 0; off < groups; off += 65535u * 32u) {
    const size_t n = std::min<size_t>(groups - off, 65535u * 32u);
    dkg::small_prime_sieve_kernel<<<(unsigned)n, 128, 0, d->stream>>>(d_mod + off * limbs, limbs, n, d_pr, nprimes, d_fl + off);
    g_launches.fetch_add(1);
  }
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(flags, d_fl, groups, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  return DKG_OK;
}

// ok[g] = 1 iff every one of the `correct` tests of candidate g satisfies v_1 = +- prod_{i>1} v_i
extern "C" int dkg_biprime_verdict(int device, const uint32_t* moduli, const uint32_t* v, int parties, int correct,
                                   uint8_t* ok, size_t groups, int limbs) {
  if (!moduli || !v || !ok || parties < 1 || correct <= 0 || limbs <= 0) return fail(DKG_ERR_INVALID, "null/empty argument");
  if (limbs > dkg::kGroupedMaxLimbs) return fail(DKG_ERR_UNSUPPORTED, "candidate wider than the biprime kernels support");
  if (groups == 0) return DKG_OK;
  for (size_t g = 0; g < groups; ++g)
    if ((moduli[g * (size_t)limbs] & 1u) == 0) return fail(DKG_ERR_INVALID, "every modulus must be odd");
  DeviceState* d = nullptr;
  int rc = device_state(device, &d);
  if (rc != DKG_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  DeviceLease lease(d, d->stream);
  DevBufs bufs(d->stream);
  uint32_t *d_mod, *d_v, *d_ok;
  const size_t mod_b = groups * (size_t)limbs * 4, v_b = (size_t)parties * groups * correct * limbs * 4;
  cudaError_t e = bufs.alloc(&d_mod, mod_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_v, v_b);
  if (e == cudaSuccess) e = bufs.alloc(&d_ok, groups * 4);
  if (e != cudaSuccess) return fail(DKG_ERR_NOMEM, std::string("verdict cudaMalloc: ") + cudaGetErrorString(e));
  std::vector<uint32_t> ones(groups, 1u), res(groups);
  CUDA_TRY(cudaMemcpyAsync(d_mod, moduli, mod_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_v, v, v_b, cudaMemcpyHostToDevice, d->stream));
  CUDA_TRY(cudaMemcpyAsync(d_ok, ones.data(), groups * 4, cudaMemcpyHostToDevice, d->stream));
  const unsigned long long n = groups * (unsigned long long)correct;
  dkg::biprime_verdict_kernel<<<(unsigned)((n + 63) / 64), 64, 0, d->stream>>>(d_mod, d_v, limbs, groups, parties, correct, d_ok);
  g_launches.fetch_add(1);
  CUDA_TRY(cudaGetLastError());
  CUDA_TRY(cudaMemcpyAsync(res.data(), d_ok, groups * 4, cudaMemcpyDeviceToHost, d->stream));
  CUDA_TRY(cudaStreamSynchronize(d->stream));
  for (size_t g = 0; g < groups; ++g) ok[g] = (uint8_t)(res[g] ? 1 : 0);
  return DKG_OK;
}

// ---- one call, several GPUs: in-process threshold decryption --------------------------------------
// SURVEY.md section 8(e): ciphertexts are independent, so a batch shards by index across the GPUs of
// one box -- one host thread + two streams per device, H2D of each shard from the caller's array,
// results D2H into disjoint slices of the caller's arrays (the "host gather").  No inter-GPU
// collective.  With all parties' keys in one process (DistributedPaillier with distributed=False,
// the reference's test and benchmark set-up, distributed_keygen.py:203-226) the d+1 partial
// decryptions and the combination of _decrypt_sequence_raw (:463-466, :510-515) run back to back on
// the device: the ciphertexts are uploaded once, the partials never visit the host unless asked for.

struct dkg_threshold_ctx {
  struct Dev {
    DeviceState* dev = nullptr;
    std::vector<dkg_modexp_ctx*> parties;
    dkg_combine_ctx* combine = nullptr;
    cudaStream_t streams[2] = {nullptr, nullptr};
    // shared squaring chain (modexp_nsq_multi_kernel): right-to-left digits of every party
    dkg::NsqMultiFn multi_kernel = nullptr;
    uint8_t* d_digits = nullptr;     // [shares][multi_nwin]
    int multi_w = 0, multi_nwin = 0;
    size_t multi_scratch_per_warp = 0, multi_q_offset = 0;
  };
  int shares = 0, n_limbs = 0, l2 = 0;
  size_t chunk_rows = 1 << 18;
  std::vector<Dev> devs;
};

namespace {

struct Shard { size_t lo, hi; };
std::vector<Shard> shard_rows(size_t count, size_t parts) {
  std::vector<Shard> out(parts);
  for (size_t r = 0; r < parts; ++r) out[r] = Shard{count * r / parts, count * (r + 1) / parts};
  return out;
}

// All parties' exponentiations of `rows` ciphertexts through ONE squaring chain (dkg_nsq.cuh,
// modexp_nsq_multi_kernel): entry -> multi kernel -> exit for every party; a party with a negative
// exponent gets the batched inversion applied to its RESULTS, (c^-1)^|e| = (c^|e|)^-1 (same canonical
// residue), and if a chain of that inversion met a non-unit the party's direct kernel redoes its
// rows on the same stream, predicated on the device-side flag, with the exact per-element status.
// d_part: [S][rows][l2], d_st: [S][rows].
int launch_threshold_multi(dkg_threshold_ctx::Dev& dv, int S, const uint32_t* d_bases, uint32_t* d_part, uint8_t* d_st,
                           size_t rows, cudaStream_t stream) {
  dkg_modexp_ctx* c0 = dv.parties[0];
  DeviceState* d = dv.dev;
  CUDA_TRY(cudaSetDevice(d->device));
  const int Lp = c0->nLp, l2 = c0->limbs;
  const size_t pair_words = rows * (size_t)(2 * Lp);
  // negative exponents: the party's RESULTS are inverted inside the kernel (pair_invert, exact
  // per-element status, DKG_INKERNEL_INVERSE=1) or by the batched inversion behind it
  const bool inv_in_kernel = c0->nsq_inv;
  unsigned int negative_mask = 0;
  size_t inv_words = 0, scratch_words = (size_t)c0->ctas * c0->nwarps * dv.multi_scratch_per_warp;
  for (int p = 0; p < S; ++p) {
    const dkg_modexp_ctx* c = dv.parties[p];
    if (c->negative && inv_in_kernel) negative_mask |= 1u << p;
    if (!c->negative || inv_in_kernel) continue;
    inv_words = batchinv_area(c, rows);   // the same for every party (one N)
    scratch_words = std::max(scratch_words, (size_t)c->ctas * c->warps * c->scratch_per_warp);   // its direct redo
  }
  int rc = ensure_aux(d, inv_words + (size_t)(S + 1) * pair_words);
  if (rc == DKG_OK) rc = ensure_scratch(d, scratch_words);
  if (rc != DKG_OK) return rc;
  uint32_t* pairs_in = d->aux + inv_words;
  uint32_t* pairs_out = pairs_in + pair_words;
  CUDA_TRY(cudaMemsetAsync(d_st, 0, rows * (size_t)S, stream));
  dkg::NsqIoParams e{};
  e.in = d_bases; e.out = pairs_in; e.count = rows; e.io_limbs = l2; e.Lp = Lp; e.consts = c0->d_nio; e.n0inv = c0->n_n0inv;
  e.mrows = nullptr; e.m_limbs = 0;
  dkg::nsq_entry_kernel<<<(unsigned)((rows + 63) / 64), 64, 0, stream>>>(e);
  CUDA_TRY(cudaMemsetAsync(d->counter, 0, sizeof(unsigned int), stream));
  dkg::NsqMultiParams q{};
  q.pairs_in = pairs_in; q.pairs_out = pairs_out; q.count = rows; q.consts = c0->d_nconsts; q.digits = dv.d_digits;
  q.nparties = S; q.nwin = dv.multi_nwin; q.wbits = dv.multi_w; q.scratch = d->scratch;
  q.negative_mask = negative_mask; q.status = d_st;
  q.scratch_per_warp = dv.multi_scratch_per_warp; q.scratch_q_offset = dv.multi_q_offset; q.counter = d->counter;
  {
    KernelTimer kt(d, stream);
    dv.multi_kernel<<<wave_ctas(c0->ctas, c0->nwarps, rows), c0->nwarps * 32, c0->nsmem, stream>>>(q);
  }
  dkg::NsqIoParams x = e;
  x.in = pairs_out; x.out = d_part; x.count = rows * (size_t)S;
  dkg::nsq_exit_kernel<<<(unsigned)((x.count + 63) / 64), 64, 0, stream>>>(x);
  CUDA_TRY(cudaGetLastError());
  g_launches.fetch_add(3);
  for (int p = 0; p < S; ++p) {
    dkg_modexp_ctx* c = dv.parties[p];
    uint32_t* out_p = d_part + (size_t)p * rows * l2;
    if (c->negative && !inv_in_kernel) {
      dkg::BatchInvParams inv;
      rc = launch_batchinv(c, out_p, rows, out_p, stream, &inv);
      if (rc == DKG_OK) rc = launch_direct(c, d_bases, out_p, d_st + (size_t)p * rows, nullptr, rows, stream, nullptr, inv.any_bad);
      if (rc != DKG_OK) return rc;
    }
    rc = launch_range_check(c, d_bases, out_p, d_st + (size_t)p * rows, rows, stream);
    if (rc != DKG_OK) return rc;
  }
  return DKG_OK;
}

// Every party's partial decryption of `rows` ciphertexts on one device, d_part: [S][rows][l2],
// d_st: [S][rows].  A few ciphertexts: every party's exponentiation in ONE cooperative launch (one
// warp per (party, ciphertext)); otherwise the shared squaring chain, else one call per party.
int launch_partials(const dkg_threshold_ctx* t, dkg_threshold_ctx::Dev& dv, const uint32_t* d_in, uint32_t* d_part,
                    uint8_t* d_st, size_t rows, cudaStream_t s) {
  const int S = t->shares;
  bool fused = S <= dkg::kCoopMaxParties;
  for (int p = 0; p < S; ++p) fused = fused && dv.parties[p]->coop && rows * (size_t)S <= dv.parties[p]->coop_max;
  int rc = DKG_OK;
  if (fused) {
    rc = launch_modexp_coop_parties(dv.parties.data(), S, d_in, d_part, d_st, rows, s, nullptr, 0);
    for (int p = 0; p < S && rc == DKG_OK; ++p)
      rc = launch_range_check(dv.parties[p], d_in, d_part + (size_t)p * rows * t->l2, d_st + (size_t)p * rows, rows, s);
    return rc;
  }
  if (dv.multi_kernel != nullptr) {
    rc = launch_threshold_multi(dv, S, d_in, d_part, d_st, rows, s);
    if (rc != DKG_ERR_NOMEM) return rc;
    dv.multi_kernel = nullptr;   // no room for the bucket scratch: one exponentiation per party from here on
    rc = DKG_OK;
  }
  for (int p = 0; p < S && rc == DKG_OK; ++p)
    rc = launch_modexp(dv.parties[p], d_in, d_part + (size_t)p * rows * t->l2, d_st + (size_t)p * rows, rows, s);
  return rc;
}

// what one device does with its shard, chunk by chunk, alternating between its two streams so the
// copies of one chunk overlap the kernels of the other.  mode 0: decrypt (partials optional),
// 1: one party's partial decryption, 2: combination of given partials, 3: every party's partial
// decryptions without the combination (status per party, [shares][count]).
struct ThresholdJob {
  int mode = 0, party = 0;
  const uint32_t* in = nullptr;        // mode 0/1: ciphertexts [count][l2]; mode 2: partials [shares][count][l2]
  uint32_t* plain = nullptr;           // [count][n_limbs]  (mode 0/2)
  uint32_t* partials = nullptr;        // mode 0: optional [shares][count][l2]; mode 1: [count][l2]
  uint8_t* status = nullptr;           // [count] or null
  size_t count = 0;                    // rows of the whole call (stride between shares)
};

int run_threshold_shard(dkg_threshold_ctx* t, dkg_threshold_ctx::Dev& dv, const ThresholdJob& job, Shard sh, std::string* err) {
  auto failed = [&](int code, const std::string& msg) { *err = msg; return code; };
#define TRY_CUDA(expr)                                                                            \
  do {                                                                                            \
    cudaError_t e__ = (expr);                                                                     \
    if (e__ != cudaSuccess) return failed(DKG_ERR_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
  } while (0)
  if (sh.hi <= sh.lo) return DKG_OK;
  TRY_CUDA(cudaSetDevice(dv.dev->device));
  const int S = t->shares, l2 = t->l2, ln = t->n_limbs;
  const size_t rows_max = std::min(t->chunk_rows, sh.hi - sh.lo);
  const size_t row_b = (size_t)l2 * 4, plain_b = (size_t)ln * 4;
  struct Buf { uint32_t *in = nullptr, *part = nullptr, *out = nullptr; uint8_t* st = nullptr; std::vector<uint8_t> host_st; size_t lo = 0, rows = 0; bool busy = false; } buf[2];
  const bool need_part = job.mode != 1;       // [S][rows][l2] on the device
  for (int b = 0; b < 2; ++b) {
    cudaStream_t s = dv.streams[b];
    if (job.mode != 2) TRY_CUDA(cudaMallocAsync(&buf[b].in, rows_max * row_b, s));
    TRY_CUDA(cudaMallocAsync(&buf[b].part, rows_max * row_b * (need_part ? S : 1), s));
    if (job.mode != 1 && job.mode != 3) TRY_CUDA(cudaMallocAsync(&buf[b].out, rows_max * plain_b, s));
    TRY_CUDA(cudaMallocAsync(&buf[b].st, rows_max * (size_t)(S + 1), s));
    buf[b].host_st.resize(rows_max * (size_t)(S + 1));
  }
  auto finish = [&](Buf& B, cudaStream_t s) -> int {
    if (!B.busy) return DKG_OK;
    TRY_CUDA(cudaStreamSynchronize(s));
    B.busy = false;
    if (job.status) {
      for (size_t i = 0; i < B.rows; ++i) {
        uint8_t st = 0;
        if (job.mode == 3) {
          for (int p = 0; p < S; ++p) job.status[(size_t)p * job.count + B.lo + i] = B.host_st[(size_t)p * B.rows + i];
          continue;
        }
        if (job.mode == 1) st = B.host_st[i];
        else {
          if (job.mode == 0)
            for (int p = 0; p < S && st == 0; ++p) st = B.host_st[(size_t)p * B.rows + i];
          if (st == 0) st = B.host_st[(size_t)S * B.rows + i];
        }
        job.status[B.lo + i] = st;
      }
    }
    return DKG_OK;
  };
  int which = 0, rc = DKG_OK;
  for (size_t lo = sh.lo; lo < sh.hi && rc == DKG_OK; lo += rows_max, which ^= 1) {
    Buf& B = buf[which];
    cudaStream_t s = dv.streams[which];
    rc = finish(B, s);
    if (rc != DKG_OK) break;
    const size_t rows = std::min(rows_max, sh.hi - lo);
    B.lo = lo; B.rows = rows; B.busy = true;
    if (job.mode == 2) {
      for (int p = 0; p < S; ++p)
        TRY_CUDA(cudaMemcpyAsync(B.part + (size_t)p * rows * l2, job.in + ((size_t)p * job.count + lo) * l2, rows * row_b, cudaMemcpyHostToDevice, s));
    } else {
      TRY_CUDA(cudaMemcpyAsync(B.in, job.in + lo * l2, rows * row_b, cudaMemcpyHostToDevice, s));
    }
    {
      DeviceLease lease(dv.dev, s);
      if (job.mode == 1) {
        rc = launch_modexp(dv.parties[job.party], B.in, B.part, B.st, rows, s);
      } else {
        if (job.mode == 0 || job.mode == 3) rc = launch_partials(t, dv, B.in, B.part, B.st, rows, s);
        if (rc == DKG_OK && job.mode != 3) rc = launch_combine(dv.combine, B.part, B.out, B.st + (size_t)S * rows, rows, s);
      }
      if (rc != DKG_OK) { *err = g_err; break; }
    }
    if (job.mode == 1) {
      TRY_CUDA(cudaMemcpyAsync(job.partials + lo * l2, B.part, rows * row_b, cudaMemcpyDeviceToHost, s));
      if (job.status) TRY_CUDA(cudaMemcpyAsync(B.host_st.data(), B.st, rows, cudaMemcpyDeviceToHost, s));
    } else {
      if (job.mode != 3) TRY_CUDA(cudaMemcpyAsync(job.plain + lo * ln, B.out, rows * plain_b, cudaMemcpyDeviceToHost, s));
      if ((job.mode == 0 || job.mode == 3) && job.partials)
        for (int p = 0; p < S; ++p)
          TRY_CUDA(cudaMemcpyAsync(job.partials + ((size_t)p * job.count + lo) * l2, B.part + (size_t)p * rows * l2, rows * row_b, cudaMemcpyDeviceToHost, s));
      if (job.status) TRY_CUDA(cudaMemcpyAsync(B.host_st.data(), B.st, rows * (size_t)(S + 1), cudaMemcpyDeviceToHost, s));
    }
  }
  for (int b = 0; b < 2; ++b) {
    const int r2 = finish(buf[b], dv.streams[b]);
    if (rc == DKG_OK) rc = r2;
    cudaStream_t s = dv.streams[b];
    if (buf[b].in) cudaFreeAsync(buf[b].in, s);
    if (buf[b].part) cudaFreeAsync(buf[b].part, s);
    if (buf[b].out) cudaFreeAsync(buf[b].out, s);
    if (buf[b].st) cudaFreeAsync(buf[b].st, s);
  }
  return rc;
#undef TRY_CUDA
}

int run_threshold(dkg_threshold_ctx* t, const ThresholdJob& job) {
  if (job.count == 0) return DKG_OK;
  const size_t ndev = t->devs.size();
  const std::vector<Shard> shards = shard_rows(job.count, ndev);
  std::vector<int> rcs(ndev, DKG_OK);
  std::vector<std::string> errs(ndev);
  std::vector<std::thread> threads;
  for (size_t r = 1; r < ndev; ++r)
    threads.emplace_back([&, r] { rcs[r] = run_threshold_shard(t, t->devs[r], job, shards[r], &errs[r]); });
  rcs[0] = run_threshold_shard(t, t->devs[0], job, shards[0], &errs[0]);
  for (auto& th : threads) th.join();
  for (size_t r = 0; r < ndev; ++r)
    if (rcs[r] != DKG_OK) return fail(rcs[r], "device " + std::to_string(t->devs[r].dev->device) + ": " + errs[r]);
  return DKG_OK;
}

// Shared squaring chain for a device's parties (launch_threshold_multi): eligible when there are at
// least two of them, all on the pair arithmetic with one shape, table access not in constant-time
// mode, and the batched inversion available if an exponent is negative.  Window width: fewest
// multiplications per party, ceil(E / w) + 2 (2^w - 2), under a cap on the bucket scratch.
int setup_threshold_multi(dkg_threshold_ctx::Dev& dv, int shares, const uint32_t* exponents, int exp_limbs) {
  if (shares < 2 || shares > dkg::kNsqMultiMaxParties || env_long("DKG_SHARED_SQUARINGS", 1) == 0) return DKG_OK;
  const dkg_modexp_ctx* c0 = dv.parties[0];
  int ebits = 1;
  for (int p = 0; p < shares; ++p) {
    const dkg_modexp_ctx* c = dv.parties[p];
    if (!c->nsq || c->ct_table || c->nshape.K != c0->nshape.K || c->nshape.M != c0->nshape.M || c->nsq_bg != c0->nsq_bg) return DKG_OK;
    if (c->negative && c->inv_kernel == nullptr) return DKG_OK;
    ebits = std::max(ebits, c->ebits);
  }
  const dkg::ShapeKernels kernels = lookup_kernels(c0->nshape.K, c0->nshape.M);
  const dkg::NsqMultiFn kernel = c0->nsq_bg ? kernels.multi_bg : kernels.multi;
  if (!kernel) return DKG_OK;
  const size_t slot_words = (size_t)2 * c0->nLs * 32;   // one pair in lane layout
  const size_t total_warps = (size_t)c0->ctas * c0->nwarps;
  const size_t cap_words = (size_t)env_long("DKG_MULTI_SCRATCH_MB", 24576) * (1u << 18);
  int best = 0;
  long best_cost = -1;
  for (int w = 1; w <= 8; ++w) {
    const size_t words = total_warps * (((size_t)shares << w) + 2 + 4) * slot_words;
    if (w > 1 && words > cap_words) break;
    const long cost = (ebits + w - 1) / w + 2 * ((1L << w) - 2);
    if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = w; }
  }
  if (long f = env_long("DKG_MULTI_WINDOW", 0); f >= 1 && f <= 8) best = (int)f;
  const int w = best, nwin = (ebits + w - 1) / w;
  std::vector<uint8_t> digits((size_t)shares * nwin, 0);
  for (int p = 0; p < shares; ++p) {
    const uint32_t* e = exponents + (size_t)p * exp_limbs;
    for (int k = 0; k < nwin; ++k) {
      unsigned dgt = 0;
      for (int b = 0; b < w; ++b) {
        const int bit = k * w + b;
        if (bit < 32 * exp_limbs && ((e[bit / 32] >> (bit % 32)) & 1u)) dgt |= 1u << b;
      }
      digits[(size_t)p * nwin + k] = (uint8_t)dgt;
    }
  }
  CUDA_TRY(cudaSetDevice(dv.dev->device));
  CUDA_TRY(cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c0->nsmem));
  CUDA_TRY(cudaMalloc(&dv.d_digits, digits.size()));
  CUDA_TRY(cudaMemcpy(dv.d_digits, digits.data(), digits.size(), cudaMemcpyHostToDevice));
  dv.multi_w = w; dv.multi_nwin = nwin;
  dv.multi_q_offset = (((size_t)shares << w) + 2 + 4) * slot_words;   // buckets | parked power | accumulator | inversion work space
  dv.multi_scratch_per_warp = dv.multi_q_offset + (size_t)c0->nLs * 32 * (c0->nsq_bg ? 2 : 1);   // Q [| b]
  dv.multi_kernel = kernel;
  return DKG_OK;
}

}  // namespace

extern "C" {

int dkg_threshold_ctx_create(const int* devices, int ndev, const uint32_t* n, int n_limbs, const uint32_t* theta_inv,
                             int shares, const uint32_t* exponents, int exp_limbs, const uint8_t* negative,
                             dkg_threshold_ctx** out) {
  if (!devices || ndev <= 0 || !n || !theta_inv || !exponents || !negative || !out || shares < 1 || exp_limbs <= 0 || n_limbs <= 0)
    return fail(DKG_ERR_INVALID, "null/empty argument");
  auto* t = new dkg_threshold_ctx();
  t->shares = shares;
  if (long c = env_long("DKG_CHUNK_ROWS", 0); c > 0) t->chunk_rows = (size_t)c;
  for (int i = 0; i < ndev; ++i) {
    dkg_threshold_ctx::Dev dv;
    int rc = device_state(devices[i], &dv.dev);
    for (int p = 0; p < shares && rc == DKG_OK; ++p) {
      dkg_modexp_ctx* c = nullptr;
      rc = dkg_modexp_ctx_create_nsq(devices[i], n, n_limbs, exponents + (size_t)p * exp_limbs, exp_limbs, negative[p], &c);
      if (rc == DKG_OK) dv.parties.push_back(c);
    }
    if (rc == DKG_OK) rc = dkg_combine_ctx_create(devices[i], n, n_limbs, theta_inv, shares, &dv.combine);
    if (rc == DKG_OK) rc = setup_threshold_multi(dv, shares, exponents, exp_limbs);
    if (rc == DKG_OK) {
      cudaSetDevice(devices[i]);
      for (int b = 0; b < 2 && rc == DKG_OK; ++b)
        if (cudaStreamCreateWithFlags(&dv.streams[b], cudaStreamNonBlocking) != cudaSuccess) rc = fail(DKG_ERR_CUDA, "stream creation failed");
    }
    t->devs.push_back(dv);
    if (rc != DKG_OK) { const std::string keep = g_err; dkg_threshold_ctx_destroy(t); g_err = keep; return rc; }
  }
  t->n_limbs = t->devs[0].combine->ln;
  t->l2 = t->devs[0].combine->l2;
  if (env_long("DKG_CHUNK_ROWS", 0) <= 0) {
    // chunks of whole kernel waves (4 of them): no partially filled last wave inside a shard
    const dkg_modexp_ctx* c = t->devs[0].parties[0];
    const size_t wave = (size_t)c->ctas * (size_t)(c->nsq ? c->nwarps : c->warps) * 32;
    t->chunk_rows = std::max<size_t>(4 * wave, 1 << 16);
  }
  *out = t;
  return DKG_OK;
}

void dkg_threshold_ctx_destroy(dkg_threshold_ctx* t) {
  if (!t) return;
  for (auto& dv : t->devs) {
    if (dv.dev) cudaSetDevice(dv.dev->device);
    for (auto* c : dv.parties) dkg_modexp_ctx_destroy(c);
    dkg_combine_ctx_destroy(dv.combine);
    for (auto s : dv.streams) if (s) cudaStreamDestroy(s);
    if (dv.d_digits) cudaFree(dv.d_digits);
  }
  delete t;
}

int dkg_threshold_info(const dkg_threshold_ctx* t, int info[4]) {
  if (!t || !info) return fail(DKG_ERR_INVALID, "null argument");
  info[0] = (int)t->devs.size(); info[1] = t->shares; info[2] = t->n_limbs; info[3] = t->l2;
  return DKG_OK;
}

int dkg_threshold_info_ex(const dkg_threshold_ctx* t, int info[8]) {
  if (!t || !info) return fail(DKG_ERR_INVALID, "null argument");
  const dkg_threshold_ctx::Dev& dv = t->devs[0];
  info[0] = dv.multi_kernel != nullptr ? 1 : 0; info[1] = dv.multi_w; info[2] = dv.multi_nwin;
  info[3] = dv.parties[0]->nshape.K; info[4] = dv.parties[0]->nshape.M; info[5] = dv.parties[0]->nwarps;
  info[6] = dv.parties[0]->ctas; info[7] = (int)std::min<size_t>(t->chunk_rows, 0x7fffffff);
  return DKG_OK;
}

int dkg_threshold_decrypt_batch(dkg_threshold_ctx* t, const uint32_t* ciphertexts, uint32_t* plaintexts, uint32_t* partials,
                                uint8_t* status, size_t count) {
  if (!t || (count && (!ciphertexts || !plaintexts))) return fail(DKG_ERR_INVALID, "null argument");
  ThresholdJob job;
  job.mode = 0; job.in = ciphertexts; job.plain = plaintexts; job.partials = partials; job.status = status; job.count = count;
  return run_threshold(t, job);
}

// Device-resident variant on the context's FIRST device: everything already in HBM, enqueued on the
// caller's stream, no copies, no synchronisation.
int dkg_threshold_decrypt_batch_device(dkg_threshold_ctx* t, const uint32_t* d_ciphertexts, uint32_t* d_plaintexts,
                                       uint32_t* d_partials, uint8_t* d_status, size_t count, void* stream) {
  if (!t || (count && (!d_ciphertexts || !d_plaintexts || !d_partials || !d_status))) return fail(DKG_ERR_INVALID, "null argument");
  if (count == 0) return DKG_OK;
  dkg_threshold_ctx::Dev& dv = t->devs[0];
  cudaStream_t s = (cudaStream_t)stream;
  const int S = t->shares;
  DeviceLease lease(dv.dev, s);
  int rc = launch_partials(t, dv, d_ciphertexts, d_partials, d_status, count, s);
  if (rc == DKG_OK) rc = launch_combine(dv.combine, d_partials, d_plaintexts, d_status + (size_t)S * count, count, s);
  return rc;
}

int dkg_threshold_partial_decrypt_batch(dkg_threshold_ctx* t, int party, const uint32_t* ciphertexts, uint32_t* out,
                                        uint8_t* status, size_t count) {
  if (!t || party < 0 || party >= t->shares || (count && (!ciphertexts || !out))) return fail(DKG_ERR_INVALID, "bad argument");
  ThresholdJob job;
  job.mode = 1; job.party = party; job.in = ciphertexts; job.partials = out; job.status = status; job.count = count;
  return run_threshold(t, job);
}

int dkg_threshold_partials_batch(dkg_threshold_ctx* t, const uint32_t* ciphertexts, uint32_t* partials, uint8_t* status, size_t count) {
  if (!t || (count && (!ciphertexts || !partials))) return fail(DKG_ERR_INVALID, "null argument");
  ThresholdJob job;
  job.mode = 3; job.in = ciphertexts; job.partials = partials; job.status = status; job.count = count;
  return run_threshold(t, job);
}

int dkg_threshold_combine_batch(dkg_threshold_ctx* t, const uint32_t* partials, uint32_t* plaintexts, uint8_t* status, size_t count) {
  if (!t || (count && (!partials || !plaintexts))) return fail(DKG_ERR_INVALID, "null argument");
  ThresholdJob job;
  job.mode = 2; job.in = partials; job.plain = plaintexts; job.status = status; job.count = count;
  return run_threshold(t, job);
}

/* page-lock / release a caller buffer so that the copies above run at full PCIe rate */
int dkg_host_register(void* ptr, size_t bytes) {
  if (!ptr || !bytes) return fail(DKG_ERR_INVALID, "null argument");
  CUDA_TRY(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
  return DKG_OK;
}
int dkg_host_unregister(void* ptr) {
  if (!ptr) return fail(DKG_ERR_INVALID, "null argument");
  CUDA_TRY(cudaHostUnregister(ptr));
  return DKG_OK;
}

}  // extern "C"
