// fp32 CUDA-core kernels of the HiFi-GAN-NSF generator on the G32T activation layout (common.cuh).
//
// conv1d_c4_ffma: implicit-GEMM 1-D convolution.  CTA tile = 256 time rows x (8 warps * CPT) output
// columns; lanes run along time (consecutive 16-byte rows -> conflict-free LDS.128 and coalesced
// 128-bit global access), warps run along output channels (weight reads are warp broadcasts).
// Input channels are consumed 16 at a time through shared memory; the leaky-relu pre-activation
// of the ResBlocks (hifigan.py:55,57) is applied while staging, bias / residual / 1/num_kernels
// scaling / ResBlock-sum accumulation are fused in the epilogue.
#include <algorithm>

#include "conv_ffma.cuh"

namespace svb {

constexpr int kRowsPerThread = 8;   // 8 rows x 32 lanes = 256-row tile
constexpr int kCK = 16;             // input channels per shared-memory chunk

template <int KS, int CPT>
__global__ void __launch_bounds__(256) conv1d_c4_ffma_kernel(ConvArgs a) {
    extern __shared__ float4 smem4[];
    constexpr int CO_TILE = 8 * CPT;
    const int halo = (KS - 1) / 2 * a.dil;
    const int rows = kTileT + 2 * halo;
    float4 *xs = smem4;                                        // [4 quads][rows]
    float *ws = reinterpret_cast<float *>(smem4 + 4 * rows);   // [KS][kCK][CO_TILE]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b = blockIdx.z;
    const int t0 = blockIdx.x * kTileT;
    const int co_tile0 = blockIdx.y * CO_TILE;
    const int co0 = co_tile0 + warp * CPT;                     // first GEMM column of this warp
    const bool active = co0 < a.CoutP;
    const int cin_q = a.Cin >> 2;
    const int Tq = valid_rows(a, b);
    if (t0 >= Tq) return;                                      // tile wholly past this clip's end (ragged batch)

    float acc[kRowsPerThread][CPT];
#pragma unroll
    for (int r = 0; r < kRowsPerThread; ++r)
#pragma unroll
        for (int c = 0; c < CPT; ++c) acc[r][c] = 0.f;

    const float4 *in4 = reinterpret_cast<const float4 *>(a.in);

    for (int c0 = 0; c0 < a.Cin; c0 += kCK) {
        __syncthreads();
        // ---- stage the activation slab: 4 quads x rows, pre-activation fused
        for (int idx = tid; idx < 4 * rows; idx += 256) {
            const int q = idx & 3, r = idx >> 2;            // the 4 quads of a row are 64 contiguous bytes
            const int cq = (c0 >> 2) + q;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (cq < cin_q) {
                v = __ldg(in4 + act_q4(b, a.Cin, a.in_Tp, cq, kPad + t0 - halo + r));
                v = lrelu4(v, a.in_slope);
            }
            xs[q * rows + r] = v;
        }
        // ---- stage the weight chunk [KS][kCK][CO_TILE]
        for (int idx = tid; idx < KS * kCK * (CO_TILE / 4); idx += 256) {
            const int co4 = idx % (CO_TILE / 4);
            const int ci = (idx / (CO_TILE / 4)) % kCK;
            const int k = idx / (CO_TILE / 4 * kCK);
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int co = co_tile0 + co4 * 4;
            if (c0 + ci < a.Cin && co < a.CoutP)
                v = __ldg(reinterpret_cast<const float4 *>(a.w + ((size_t)k * a.Cin + c0 + ci) * a.CoutP + co));
            reinterpret_cast<float4 *>(ws)[idx] = v;
        }
        __syncthreads();
        if (!active) continue;
        const int nq = min(4, cin_q - (c0 >> 2));
#pragma unroll 1
        for (int q = 0; q < nq; ++q) {
#pragma unroll
            for (int k = 0; k < KS; ++k) {
                float4 xv[kRowsPerThread];
#pragma unroll
                for (int r = 0; r < kRowsPerThread; ++r) xv[r] = xs[q * rows + lane + 32 * r + k * a.dil];
#pragma unroll
                for (int ci = 0; ci < 4; ++ci) {
                    const float *wp = ws + ((k * kCK + q * 4 + ci) * CO_TILE) + warp * CPT;
                    float wv[CPT];
#pragma unroll
                    for (int c4 = 0; c4 < CPT / 4; ++c4) {
                        const float4 w4 = *reinterpret_cast<const float4 *>(wp + 4 * c4);
                        wv[4 * c4 + 0] = w4.x, wv[4 * c4 + 1] = w4.y, wv[4 * c4 + 2] = w4.z, wv[4 * c4 + 3] = w4.w;
                    }
#pragma unroll
                    for (int r = 0; r < kRowsPerThread; ++r) {
                        const float x = ci == 0 ? xv[r].x : ci == 1 ? xv[r].y : ci == 2 ? xv[r].z : xv[r].w;
#pragma unroll
                        for (int c = 0; c < CPT; ++c) acc[r][c] = fmaf(x, wv[c], acc[r][c]);
                    }
                }
            }
        }
    }
    if (!active) return;

    // ---- epilogue
#pragma unroll
    for (int c4 = 0; c4 < CPT / 4; ++c4) {
        const int cop = co0 + 4 * c4;                 // GEMM column of this quad
        if (cop >= a.CoutP) break;
        int phi = 0, co = cop;
        if (a.ups_u > 0) { phi = cop / a.Cout; co = cop - phi * a.Cout; }
        const float4 bv = a.bias ? __ldg(reinterpret_cast<const float4 *>(a.bias + co)) : make_float4(0, 0, 0, 0);
#pragma unroll
        for (int r = 0; r < kRowsPerThread; ++r) {
            const int q = t0 + lane + 32 * r;
            if (q >= Tq) continue;
            const size_t row = act_q4(b, a.Cout, a.out_Tp, co >> 2, kPad + (a.ups_u > 0 ? q * a.ups_u + phi : q));
            float4 v = make_float4(acc[r][4 * c4 + 0] + bv.x, acc[r][4 * c4 + 1] + bv.y,
                                   acc[r][4 * c4 + 2] + bv.z, acc[r][4 * c4 + 3] + bv.w);
            if (a.res) {
                const float4 rv = __ldg(reinterpret_cast<const float4 *>(a.res) + row);
                v.x += rv.x, v.y += rv.y, v.z += rv.z, v.w += rv.w;
            }
            v.x *= a.out_scale, v.y *= a.out_scale, v.z *= a.out_scale, v.w *= a.out_scale;
            float4 *op = reinterpret_cast<float4 *>(a.out) + row;
            if (a.accumulate) {
                const float4 o = *op;
                v.x += o.x, v.y += o.y, v.z += o.z, v.w += o.w;
            }
            *op = v;
        }
    }
}

template <int KS, int CPT>
static int launch_conv_t(const ConvArgs &a, cudaStream_t st) {
    const int halo = (KS - 1) / 2 * a.dil;
    const int rows = kTileT + 2 * halo;
    const size_t smem = (size_t)4 * rows * 16 + (size_t)KS * kCK * (8 * CPT) * 4;
    auto kern = conv1d_c4_ffma_kernel<KS, CPT>;
    static size_t configured = 0;
    if (smem > configured) {
        SVB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    dim3 grid((a.Tq + kTileT - 1) / kTileT, (a.CoutP + 8 * CPT - 1) / (8 * CPT), a.B);
    kern<<<grid, 256, smem, st>>>(a);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

int launch_conv_ffma(const ConvArgs &a, cudaStream_t st) {
    SVB_CHECK(a.Cin % 4 == 0 && a.Cout % 4 == 0 && a.CoutP % 4 == 0, SVB_ERR_INVALID,
              "conv: channels must be multiples of 4 (Cin %d Cout %d)", a.Cin, a.Cout);
    SVB_CHECK((a.KS - 1) / 2 * a.dil <= kPad, SVB_ERR_INVALID, "conv: halo %d exceeds pad %d",
              (a.KS - 1) / 2 * a.dil, kPad);
    const bool wide = (a.Cout % 8 == 0) && a.CoutP >= 64;
#define SVB_CONV_CASE(K)                                                        \
    case K:                                                                     \
        return wide ? launch_conv_t<K, 8>(a, st) : launch_conv_t<K, 4>(a, st);
    switch (a.KS) {
        SVB_CONV_CASE(1)
        SVB_CONV_CASE(3)
        SVB_CONV_CASE(5)
        SVB_CONV_CASE(7)
        SVB_CONV_CASE(9)
        SVB_CONV_CASE(11)
        default:
            set_error("conv: unsupported kernel size %d (odd sizes 1..11)", a.KS);
            return SVB_ERR_INVALID;
    }
#undef SVB_CONV_CASE
}

// ------------------------------------------------------------------------------ layout changes
__global__ void nct_to_c4t_kernel(const float *__restrict__ nct, float4 *__restrict__ c4t, int C, int T, int Tp,
                                  const int *__restrict__ len) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int cq = blockIdx.y, b = blockIdx.z;
    if (t >= T) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!len || t < len[b]) {
        const float *p = nct + ((size_t)b * C + cq * 4) * T + t;
        v = make_float4(p[0], p[T], p[2 * (size_t)T], p[3 * (size_t)T]);
    }
    c4t[act_q4(b, C, Tp, cq, kPad + t)] = v;
}

__global__ void c4t_to_nct_kernel(const float4 *__restrict__ c4t, float *__restrict__ nct, int C, int T, int Tp) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    const int cq = blockIdx.y, b = blockIdx.z;
    if (t >= T) return;
    const float4 v = c4t[act_q4(b, C, Tp, cq, kPad + t)];
    float *p = nct + ((size_t)b * C + cq * 4) * T + t;
    p[0] = v.x, p[T] = v.y, p[2 * (size_t)T] = v.z, p[3 * (size_t)T] = v.w;
}

__global__ void btc_to_c4t_kernel(const float4 *__restrict__ btc, float4 *__restrict__ c4t, int C, int T, int Tp, Ragged rg) {
    // one thread per (t, quad): reads 16 B of the frame-major row, writes one C4T row
    const int cq = blockIdx.x * blockDim.x + threadIdx.x;
    const int t = blockIdx.y, b = blockIdx.z;
    if (cq >= (C >> 2)) return;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (!rg.len || t < rg.len[b]) v = btc[((rg.off ? (size_t)rg.off[b] : (size_t)b * T) + t) * (C >> 2) + cq];
    c4t[act_q4(b, C, Tp, cq, kPad + t)] = v;
}

int launch_nct_to_c4t(const float *nct, float *c4t, int B, int C, int T, int Tp, cudaStream_t st, Ragged rg) {
    dim3 grid((T + 127) / 128, C / 4, B);
    nct_to_c4t_kernel<<<grid, 128, 0, st>>>(nct, reinterpret_cast<float4 *>(c4t), C, T, Tp, rg.len);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}
int launch_c4t_to_nct(const float *c4t, float *nct, int B, int C, int T, int Tp, cudaStream_t st) {
    dim3 grid((T + 127) / 128, C / 4, B);
    c4t_to_nct_kernel<<<grid, 128, 0, st>>>(reinterpret_cast<const float4 *>(c4t), nct, C, T, Tp);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}
int launch_btc_to_c4t(const float *btc, float *c4t, int B, int C, int T, int Tp, cudaStream_t st, Ragged rg) {
    dim3 grid((C / 4 + 31) / 32, T, B);
    btc_to_c4t_kernel<<<grid, 32, 0, st>>>(reinterpret_cast<const float4 *>(btc), reinterpret_cast<float4 *>(c4t), C,
                                           T, Tp, rg);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

// ------------------------------------------------------------------------------ NSF injection
// one thread per (row n, channel quad): the 8 quads of a 32-channel group are 8 consecutive lanes, so
// a warp touches 4 whole 128-byte rows; har[] is a broadcast within a row; nw is packed [K][C].
__global__ void noise_conv_add_kernel(float4 *__restrict__ x, int C, int T, int Tp, const float *__restrict__ har,
                                      int Thar, const float *__restrict__ nw, const float *__restrict__ nb, int K,
                                      int stride, int pad, const int *__restrict__ len, int x_mul, int har_mul) {
    const int cq_n = c4t_groups(C) * 8;                       // quads per row incl. zero padding channels
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    const int Hb = len ? len[b] * har_mul : Thar;             // har samples of this clip
    if (len) T = len[b] * x_mul;
    if (idx >= (long long)T * cq_n) return;
    const int n = (int)(idx / cq_n), cq = (int)(idx - (long long)n * cq_n);
    if (cq * 4 >= C) return;
    const float *h = har + (size_t)b * Thar;
    float4 acc = __ldg(reinterpret_cast<const float4 *>(nb) + cq);
    const int base = n * stride - pad;
    for (int j = 0; j < K; ++j) {
        const int i = base + j;
        if (i < 0 || i >= Hb) continue;
        const float hv = __ldg(h + i);
        const float4 w = __ldg(reinterpret_cast<const float4 *>(nw + (size_t)j * C) + cq);
        acc.x = fmaf(w.x, hv, acc.x), acc.y = fmaf(w.y, hv, acc.y), acc.z = fmaf(w.z, hv, acc.z), acc.w = fmaf(w.w, hv, acc.w);
    }
    float4 *p = x + act_q4(b, C, Tp, cq, kPad + n);
    float4 v = *p;
    v.x += acc.x, v.y += acc.y, v.z += acc.z, v.w += acc.w;
    *p = v;
}

int launch_noise_conv_add(float *x, int B, int C, int T, int Tp, const float *har, int Thar, const float *nw,
                          const float *nb, int K, int stride, int pad, cudaStream_t st, Ragged rg, int x_mul, int har_mul) {
    const long long total = (long long)T * c4t_groups(C) * 8;
    dim3 grid((unsigned)((total + 255) / 256), B);
    noise_conv_add_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<float4 *>(x), C, T, Tp, har, Thar, nw, nb, K, stride, pad, rg.len,
                                                x_mul, har_mul);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

// ------------------------------------------------------------------------------ conv_post + tanh
__global__ void __launch_bounds__(256) conv_post_tanh_kernel(const float4 *__restrict__ x, int C, int T, int Tp,
                                                             const float4 *__restrict__ wq, const float *__restrict__ bias, int K,
                                                             float slope, float *__restrict__ wav, Ragged rg, int mul) {
    extern __shared__ float4 sm4[];
    const int cq_n = C >> 2, halo = (K - 1) / 2, rows = 256 + 2 * halo;
    float4 *xs = sm4;               // [cq_n][rows]
    float4 *ws = sm4 + cq_n * rows; // [cq_n][K]
    const int b = blockIdx.y, t0 = blockIdx.x * 256, tid = threadIdx.x;
    // ragged batch: clip b has Tv samples; the padded output gets zeros up to T, the packed one holds the clip alone
    const int Tv = rg.len ? rg.len[b] * mul : T;
    float *wb = rg.off ? wav + (size_t)rg.off[b] * mul : wav + (size_t)b * T;
    if (!rg.off && t0 + tid >= Tv && t0 + tid < T) wb[t0 + tid] = 0.f;
    if (t0 >= Tv) return;                                   // tile wholly past the clip's end
    for (int idx = tid; idx < cq_n * rows; idx += 256) {
        const int r = idx / cq_n, cq = idx - r * cq_n;      // quads of a row are contiguous in G32T
        xs[cq * rows + r] = lrelu4(__ldg(x + act_q4(b, C, Tp, cq, kPad + t0 - halo + r)), slope);
    }
    for (int idx = tid; idx < cq_n * K; idx += 256) ws[idx] = wq[idx];
    __syncthreads();
    const int t = t0 + tid;
    if (t >= Tv) return;
    float acc = __ldg(bias);
    for (int cq = 0; cq < cq_n; ++cq)
        for (int k = 0; k < K; ++k) {
            const float4 xv = xs[cq * rows + tid + k], wv = ws[cq * K + k];
            acc = fmaf(xv.x, wv.x, acc), acc = fmaf(xv.y, wv.y, acc), acc = fmaf(xv.z, wv.z, acc),
            acc = fmaf(xv.w, wv.w, acc);
        }
    wb[t] = tanhf(acc);
}

int launch_conv_post_tanh(const float *x, int B, int C, int T, int Tp, const float *wq, const float *bias, int K, float slope,
                          float *wav, cudaStream_t st, Ragged rg, int mul) {
    const int rows = 256 + (K - 1);
    const size_t smem = (size_t)(C / 4) * (rows + K) * 16;
    SVB_CHECK(smem <= 200 * 1024, SVB_ERR_INVALID, "conv_post: %d channels do not fit shared memory", C);
    static size_t configured = 48 * 1024;
    if (smem > configured) {
        SVB_CUDA(cudaFuncSetAttribute(conv_post_tanh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    dim3 grid((T + 255) / 256, B);
    conv_post_tanh_kernel<<<grid, 256, smem, st>>>(reinterpret_cast<const float4 *>(x), C, T, Tp,
                                                   reinterpret_cast<const float4 *>(wq), bias, K, slope, wav, rg, mul);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

// ------------------------------------------------------------------------------ stale rows of a ragged batch
struct ZeroSegs {
    ZeroSeg s[kMaxZeroSegs];
};
// grid (row blocks, segment, clip): rows [len[b] * mul, hw[b] * mul) of every channel group of segment y, clip z
__global__ void zero_tails_kernel(ZeroSegs segs, const int *__restrict__ len, const int *__restrict__ hw) {
    const ZeroSeg sg = segs.s[blockIdx.y];
    const int b = blockIdx.z;
    const int r0 = len[b] * sg.mul, r1 = min(hw[b] * sg.mul, sg.Tp - 2 * kPad);
    if (r0 >= r1) return;
    const long long n = (long long)(r1 - r0) * 8 * sg.groups;             // float4s
    float4 *base = reinterpret_cast<float4 *>(sg.p);
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int q = (int)(i & 7);
        const long long rg = i >> 3;
        const int grp = (int)(rg / (r1 - r0)), r = r0 + (int)(rg - (long long)grp * (r1 - r0));
        base[(((size_t)b * sg.groups + grp) * sg.Tp + kPad + r) * 8 + q] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

int launch_zero_tails(const ZeroSeg *segs, int n, int B, const int *len, const int *hw, int max_rows, cudaStream_t st) {
    SVB_CHECK(n >= 1 && n <= kMaxZeroSegs, SVB_ERR_INVALID, "zero_tails: %d buffers (limit %d)", n, kMaxZeroSegs);
    ZeroSegs s;
    for (int i = 0; i < n; ++i) s.s[i] = segs[i];
    const dim3 grid((unsigned)std::max(1, std::min((max_rows * 8 + 255) / 256, 64)), (unsigned)n, (unsigned)B);
    zero_tails_kernel<<<grid, 256, 0, st>>>(s, len, hw);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

}  // namespace svb
