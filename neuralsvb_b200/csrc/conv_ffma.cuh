// fp32 CUDA-core kernels of the generator (conv_pre, upsamplers, NSF injection, conv_post and the
// SVB_PREC_FP32 ResBlock path).  Declarations; definitions in conv_ffma.cu.
#pragma once
#include <vector>

#include "common.cuh"

namespace svb {

// out[b][q][co'] = bias + sum_{k<KS} sum_{ci} W[k][ci][co'] * act(in[b][q + (k-(KS-1)/2)*dil][ci])
// on C4T tensors (common.cuh).  Modes:
//   residual   : + res[b][q][co']                                  (ResBlock skip, hifigan.py:59)
//   out_scale  : * s, accumulate: out += ...                        (sum of ResBlocks / num_kernels, :158-164)
//   ups_u > 0  : transposed-conv polyphase: the GEMM column co' = phi*Cout + co is stored to row
//                q*ups_u + phi, channel co of `out`                 (ConvTranspose1d, :122-125,154)
struct ConvArgs {
    const float *in;
    const float *w;       // packed [KS][Cin][CoutP]
    const float *bias;    // [Cout]
    const float *res;     // C4T like out, or nullptr
    float *out;
    int B, Cin, in_Tp;
    int Cout, out_Tp;     // channels / padded rows of the OUT tensor
    int CoutP;            // GEMM columns (= Cout, or ups_u * Cout)
    int Tq;               // valid GEMM rows q (time steps of `in`)
    int KS, dil;
    int ups_u;
    float in_slope;       // leaky-relu slope applied to `in` on load (1 = identity)
    float out_scale;
    int accumulate;
    int cin_blk = 0;      // grouped convolution (tensor-core kernel only): input channels read by ONE column block
                          // (block nblk reads channels [nblk*cin_blk, (nblk+1)*cin_blk)); 0 = dense (all Cin)
    // ragged batch: clip b has rows[b] * rows_mul valid GEMM rows (rows: device [B], in mel frames; rows_mul = the
    // upsampling factor of `in` so far).  Rows at or past that are neither computed nor stored.  nullptr: every clip Tq.
    const int *rows = nullptr;
    int rows_mul = 1;
};
__host__ __device__ inline int valid_rows(const ConvArgs &a, int b) { return a.rows ? a.rows[b] * a.rows_mul : a.Tq; }

int launch_conv_ffma(const ConvArgs &a, cudaStream_t st);

// Per-clip lengths of a ragged batch, as the element-wise kernels below take them (all device pointers, nullptr = uniform):
// clip b has len[b] frames; `off` [B + 1] = first frame of clip b in a packed (clip after clip) host-facing layout.
struct Ragged {
    const int *len = nullptr;
    const int *off = nullptr;
};

// [B][C][T] (PyTorch NCT) <-> C4T.  Ragged: rows t >= len[b] are written as zeros (the caller's padding is never read).
int launch_nct_to_c4t(const float *nct, float *c4t, int B, int C, int T, int Tp, cudaStream_t st, Ragged rg = Ragged());
int launch_c4t_to_nct(const float *c4t, float *nct, int B, int C, int T, int Tp, cudaStream_t st);
// [B][T][C] (frame-major, the reference's [T, 80] mel) -> C4T.  Ragged as above; with `off`, clip b's frames are read
// from rows off[b] .. off[b] + len[b] of a packed [sum len, C] input.
int launch_btc_to_c4t(const float *btc, float *c4t, int B, int C, int T, int Tp, cudaStream_t st, Ragged rg = Ragged());

// x[b][n][c] += nb[c] + sum_j nw[c][j] * har[b][n*stride - pad + j]     (noise_convs, hifigan.py:127-132,156-157)
// Ragged: rows n < len[b] * x_mul of x, har samples < len[b] * har_mul (the rest reads as Conv1d zero padding).
int launch_noise_conv_add(float *x, int B, int C, int T, int Tp, const float *har, int Thar, const float *nw,
                          const float *nb, int K, int stride, int pad, cudaStream_t st, Ragged rg = Ragged(), int x_mul = 1,
                          int har_mul = 1);

// wav[b][t] = tanh(bias + sum_{ci,k} w[ci][k] * lrelu(x[b][t+k-3][ci], slope))   (hifigan.py:165-167)
// Ragged: samples t >= len[b] * mul are written as 0; with `off`, clip b goes to wav[off[b] * mul ...] (packed, no tail).
int launch_conv_post_tanh(const float *x, int B, int C, int T, int Tp, const float *wq, const float *bias_dev, int K,
                          float slope, float *wav, cudaStream_t st, Ragged rg = Ragged(), int mul = 1);

// Zero the stale rows [len[b] * mul, hw[b] * mul) of G32T buffers (a ragged clip that shrank since the last call):
// seg[i] = one buffer with `groups` channel groups of Tp rows at upsampling factor `mul`.
struct ZeroSeg {
    float *p;
    int groups, Tp, mul;
};
constexpr int kMaxZeroSegs = 64;
int launch_zero_tails(const ZeroSeg *segs, int n, int B, const int *len, const int *hw, int max_rows, cudaStream_t st);

// host-side weight packing (layer_api.cu)
std::vector<float> pack_conv_weights(const float *w, int Cout, int Cin, int K);
std::vector<float> pack_convT_weights(const float *w, int Cin, int Cout, int K, int u, int pad, int *KS_out);

}  // namespace svb
