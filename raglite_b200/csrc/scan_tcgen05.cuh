// Interface of the tcgen05 / TMEM scan (RL_ALGO_TCGEN05), see scan_tcgen05.cu.
#pragma once
#include "scan_common.cuh"

namespace rl {

bool tcgen05_supported(const rl_scan_params* p);
size_t tcgen05_qimg_bytes(int B, int d);
// Builds the fp16, pre-swizzled shared-memory image of the (scaled) query batch.
int tcgen05_prepare_queries(const rl_scan_params* p, const float* q_inv_norm, float* q_scale, void* qimg,
                            cudaStream_t stream);
int launch_scan_tcgen05(const ScanArgs& a, const rl_scan_params* p, const float* q_scale, const void* qimg,
                        int sm_count, cudaStream_t stream);

}  // namespace rl
