// Instantiations and launchers of the cooperative (warp-per-operand) kernels, dkg_coop.cuh.
#include "dkg_coop.cuh"

namespace dkg {

// K = 6: up to 96 limbs per number; K = 12: up to 192.  Warps per CTA: the pair kernel runs two
// interleaved products per warp and wants the registers of a 256-thread CTA; the grouped kernel at
// K = 6 fits 16 warps.
int coop_max_warps(int K, bool pair_kernel) { return (K == 6 && !pair_kernel) ? 16 : 8; }

template <int K, int THREADS>
static cudaError_t launch_nsq_t(const CoopNsqParams& p, int ctas, int warps, size_t smem, cudaStream_t stream) {
  auto kernel = coop_nsq_kernel<K, THREADS>;
  cudaError_t e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kernel<<<ctas, warps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}
template <int K, int THREADS, bool CT>
static cudaError_t launch_grouped_t(const CoopGroupedParams& p, int ctas, int warps, size_t smem, cudaStream_t stream) {
  auto kernel = coop_grouped_kernel<K, THREADS, CT>;
  cudaError_t e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kernel<<<ctas, warps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}

template <int K, int THREADS>
static cudaError_t launch_combine_t(const CoopCombineParams& p, int ctas, int warps, size_t smem, cudaStream_t stream) {
  auto kernel = coop_combine_kernel<K, THREADS>;
  cudaError_t e = cudaFuncSetAttribute((const void*)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kernel<<<ctas, warps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}
cudaError_t launch_coop_combine(int K, const CoopCombineParams& p, int ctas, int warps, size_t smem, cudaStream_t stream) {
  if (K == 6) return launch_combine_t<6, 512>(p, ctas, warps, smem, stream);
  if (K == 12) return launch_combine_t<12, 256>(p, ctas, warps, smem, stream);
  return cudaErrorInvalidValue;
}

cudaError_t launch_coop_nsq(int K, const CoopNsqParams& p, int ctas, int warps, size_t smem, cudaStream_t stream) {
  if (K == 6) return launch_nsq_t<6, 256>(p, ctas, warps, smem, stream);
  if (K == 12) return launch_nsq_t<12, 256>(p, ctas, warps, smem, stream);
  return cudaErrorInvalidValue;
}
cudaError_t launch_coop_grouped(int K, bool ct_table, const CoopGroupedParams& p, int ctas, int warps, size_t smem,
                                cudaStream_t stream) {
  if (K == 6) return ct_table ? launch_grouped_t<6, 512, true>(p, ctas, warps, smem, stream)
                              : launch_grouped_t<6, 512, false>(p, ctas, warps, smem, stream);
  if (K == 12) return ct_table ? launch_grouped_t<12, 256, true>(p, ctas, warps, smem, stream)
                               : launch_grouped_t<12, 256, false>(p, ctas, warps, smem, stream);
  return cudaErrorInvalidValue;
}

}  // namespace dkg
