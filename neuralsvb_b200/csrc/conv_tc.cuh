// tcgen05 (5th-gen tensor core) implicit-GEMM convolution on the C4T layout.  See conv_tc.cu.
#pragma once
#include <vector>

#include "conv_ffma.cuh"

namespace svb {

struct TcWeights {
    void *blob[4] = {nullptr, nullptr, nullptr, nullptr};   // per svb_precision: weight tiles in UMMA core-matrix order
    int KS = 0, Cin = 0, CoutP = 0;
    int n_tile = 0;         // GEMM columns per CTA (UMMA N)
    bool ok = false;
};

// packed_ffma: [KS][Cin][CoutP] fp32 (the FFMA packing).  Allocations are appended to `allocs`.
// force_n_tile > 0: GEMM columns per CTA fixed by the caller (grouped layers: one tile = whole conv groups; `Cin` is then
// the number of input channels ONE column block contracts over and packed_ffma is [KS][Cin][CoutP])
int tc_pack_weights(const float *packed_ffma, int KS, int Cin, int CoutP, TcWeights *out, std::vector<void *> *allocs,
                    int force_n_tile = 0);
// same packing on the device, from a device copy of the FFMA packing into the blobs tc_pack_weights allocated
// (training: the weights change after every optimizer step)
int tc_repack_weights_dev(const float *packed_ffma_dev, const TcWeights &w, cudaStream_t st);
bool tc_supported(const TcWeights &w, const ConvArgs &a);

constexpr int kTcMaxLayers = 3;     // layers of one shape class merged into one persistent launch
// Host-built schedule of a merged launch: per CTA, the (layer, column block, clip, first row, tiles) items it executes
// in order.  chain_ordered = every CTA runs ALL layers of a tile back to back (layer 0, 1, ...): required when later
// layers accumulate into the output of earlier ones (the read-modify-write stays inside one thread); otherwise the
// items of all layers are spread over the SMs longest-processing-time first.
struct TcWorkList {
    int4 *items = nullptr;
    int *off = nullptr;
    int grid = 0, n_items = 0, MT = 0, n_layers = 0;
    bool chain_ordered = false;
    bool valid = false;             // false: rebuild before the next launch (the buffers are kept and only grow)
    size_t cap_items = 0, cap_off = 0;
};
// rows: host [B] valid GEMM rows per clip of a ragged batch (nullptr: every clip a[0].Tq); the list is uploaded on `st`
int tc_worklist_build(int n, const TcWeights *const *w, const ConvArgs *a, int precision, bool chain_ordered, TcWorkList *out,
                      const int *rows = nullptr, cudaStream_t st = 0);
void tc_worklist_free(TcWorkList *wl);
// the per-CTA item list of a merged launch is bounded (shared memory): very long batches fall back to one launch per layer
bool tc_merge_fits(int n, int B, int Tq, int Cout, int n_tile, const int *rows = nullptr);
// one persistent launch over `n` layers that share channels / rows / upsampling (taps, dilation and pointers may differ)
int launch_conv_tc_multi(int n, const TcWeights *const *w, const ConvArgs *a, int precision, cudaStream_t st, const TcWorkList &wl);
// max_ctas > 0 caps the persistent grid (used to run independent ResBlock chains side by side on SM subsets)
int launch_conv_tc(const TcWeights &w, const ConvArgs &a, int precision, cudaStream_t st, int max_ctas = 0);

}  // namespace svb
