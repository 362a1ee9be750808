// Kernel instantiations, group 0 (split across translation units so they compile in parallel).
#define DKG_GROUP 0
#define DKG_GROUP_SHAPES(X) X(16,8) X(4,1) X(4,2) X(4,3) X(8,2)
#define DKG_GROUP_GROUPED_SHAPES(X) X(16,8) X(4,1) X(4,2) X(4,3) X(8,2) X(13,5)
#define DKG_GROUP_NSQ_SHAPES(X) X(4,1) X(4,2) X(4,3) X(8,2) X(13,5)
#include "dkg_kernels.inc"

namespace dkg {
void launch_group_setup(const GroupedParams& p, bool ct_table, cudaStream_t stream) {
  const unsigned blocks = (unsigned)((p.groups + 63) / 64);
  if (ct_table) group_setup_kernel<true><<<blocks, 64, 0, stream>>>(p);
  else group_setup_kernel<false><<<blocks, 64, 0, stream>>>(p);
}
}  // namespace dkg
