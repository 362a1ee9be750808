// The kernel instantiations of one shape (K, M).  Each dkg_kernels_<n>.cu fills in the ones it
// compiled (find_kernels_group<n>); a family not instantiated for the shape stays null.
#pragma once
#include "dkg_modexp_params.h"
#include "dkg_nsq_params_fwd.h"
#include "dkg_grouped_params_fwd.h"

namespace dkg {

using KernelFn = void (*)(const ModexpParams);
using BatchInvFn = void (*)(const BatchInvParams);
using NsqFn = void (*)(const NsqParams);
using NsqMultiFn = void (*)(const NsqMultiParams);
using GroupedFn = void (*)(const GroupedParams);

struct ShapeKernels {
  KernelFn fixed = nullptr;        // modexp_fixed_kernel (direct)
  BatchInvFn batchinv = nullptr;
  NsqFn nsq = nullptr, nsq_bg = nullptr;            // pair arithmetic; _bg: b component in global scratch
  NsqMultiFn multi = nullptr, multi_bg = nullptr;   // shared squaring chain
  GroupedFn grouped = nullptr;
};

void find_kernels_group0(int K, int M, ShapeKernels* k);
void find_kernels_group1(int K, int M, ShapeKernels* k);
void find_kernels_group2(int K, int M, ShapeKernels* k);
void find_kernels_group3(int K, int M, ShapeKernels* k);
void find_kernels_group4(int K, int M, ShapeKernels* k);
void find_kernels_group5(int K, int M, ShapeKernels* k);

}  // namespace dkg
