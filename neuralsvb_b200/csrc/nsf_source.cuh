// NSF harmonic source (SineGen + SourceModuleHnNSF) on the device.  See nsf_source.cu.
#pragma once
#include "common.cuh"

namespace svb {

size_t nsf_workspace_bytes(int B, int F, int U);

// f0 [B,F] Hz (0 = unvoiced); rand_ini [B,9] / noise [B,F*U,9] or both nullptr (Philox from `seed`);
// lin_w_dev [9] / lin_b_dev [1] device (m_source.l_linear); har [B, F*U] output; sines [B, F*U, 9]
// (optional) receives the 9 harmonic signals l_linear sees, for its weight gradient.
// Ragged batch: len [B] (device) frames per clip, F = the longest; samples past len[b] * U are neither computed nor
// written and f0 / noise there is never read.  off [B + 1] (device, optional): f0 is packed clip after clip.
int launch_nsf_source(const float *f0, const float *rand_ini, const float *noise, uint64_t seed, int B, int F, int U,
                      float sr, const float *lin_w_dev, const float *lin_b_dev, void *workspace, float *har, float *sines,
                      cudaStream_t st, int *launches, const int *len = nullptr, const int *off = nullptr);

}  // namespace svb
