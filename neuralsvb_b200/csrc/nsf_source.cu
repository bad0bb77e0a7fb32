// NSF harmonic source: f0 -> tanh(Linear(9 -> 1)(SineGen(f0_upsampled))) generated on the device.
//
// Reference: HifiGanGenerator.forward lines hifigan.py:147-149 (nearest upsample of f0 by hop),
// SineGen._f02sine / forward (modules/parallel_wavegan/models/source.py:44-73,104-137) and
// SourceModuleHnNSF.forward (:385-398).
//
// The reference computes two fp32 cumsums over the whole utterance; on CPU torch accumulates
// those in double and rounds each output to float.  We reproduce that exactly without a
// sequential pass: f0 is piecewise constant per frame, so every partial sum is an integer
// combination of a few fp32 values, exactly representable in double; closed forms per frame plus
// warp scans over 32-sample chunks give bit-identical partial sums in any order.
//   S1[t] = sum_{t'<=t} rad[t']                 (phase before wrap correction, :66)
//   wrap[t] = frac(float(S1[t])) < frac(float(S1[t-1]))      (:67-68)
//   v[t]  = rad[t] + (wrap[t] ? -1 : 0)  in fp32             (:69-70,72)
//   S2[t] = sum_{t'<=t} v[t']   -> sine = sin(float(S2[t]) * 2 * pi)              (:72-73)
#include "nsf_source.cuh"

namespace svb {

constexpr int kH = 9;    // fundamental + 8 overtones (hifigan.py:112)

// ---- Philox4x32-10 (counter-based RNG for the in-kernel noise mode) ---------------------------
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0, key.y += W1;
    }
    return ctr;
}
__device__ __forceinline__ float u01(uint32_t x) { return (x >> 8) * (1.0f / 16777216.0f) + (0.5f / 16777216.0f); }
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float &n0, float &n1) {
    const float r = sqrtf(-2.0f * __logf(u01(a)));
    float s, c;
    __sincosf(6.28318530718f * u01(b), &s, &c);
    n0 = r * c, n1 = r * s;
}

__device__ __forceinline__ float rad_of(float f0, int k, float sr) {
    // f0_buf[:, :, k] = f0 * (k + 1)  (:114-118) ; rad = (f0_buf / sr) % 1  (:50)
    const float fk = (k == 0) ? f0 : f0 * (float)(k + 1);
    return fmodf(__fdiv_rn(fk, sr), 1.0f);
}

// Per-(b, k) quantities shared by all kernels.
struct NsfDims {
    int B, F, U;        // batch, frames, upsample factor (hop)
    int T;              // F * U samples
    int nchunk;         // ceil(T / 32)
    float sr;
    // ragged batch (nullptr = every clip F frames): clip b has len[b] frames; with `off`, its f0 starts at f0[off[b]]
    // (packed, clip after clip) instead of f0[b * F].  Every scan starts at t = 0 of the clip, as in a one-clip call.
    const int *len, *off;
    __device__ int frames(int b) const { return len ? len[b] : F; }
    __device__ const float *f0_of(const float *f0, int b) const { return f0 + (off ? (size_t)off[b] : (size_t)b * F); }
};

// initial phase: rand_ini[b][k] (k = 0 forced to 0, :54) or Philox uniform
__device__ __forceinline__ float rand_ini_of(const float *rand_ini, uint64_t seed, int b, int k) {
    if (k == 0) return 0.f;
    if (rand_ini) return rand_ini[b * kH + k];
    const uint4 r = philox4x32_10(make_uint4((uint32_t)b, (uint32_t)k, 0x1234u, 0u),
                                  make_uint2((uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x5eedu));
    return u01(r.x);
}

// ---- kernel 1: frame-level exclusive prefix of S1, one warp per (b, k) ------------------------
// base1[b][k][f] = S1 at the last sample before frame f, arranged so that
// S1(f, j) = base1[f] + (j + 1) * rad_f   for every sample j of frame f (incl. the very first one,
// whose value is rad_0 + rand_ini: base1[0] = fl32(rad_0 + rand_ini) - rad_0).
__global__ void nsf_frame_prefix_kernel(NsfDims d, const float *__restrict__ f0, const float *__restrict__ rand_ini,
                                        uint64_t seed, double *__restrict__ base1) {
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= d.B * kH) return;
    const int b = wid / kH, k = wid % kH;
    const float *f0b = d.f0_of(f0, b);
    const int Fb = d.frames(b);
    double *out = base1 + (size_t)wid * d.F;
    const float rad0 = rad_of(f0b[0], k, d.sr);
    const float r0p = rad0 + rand_ini_of(rand_ini, seed, b, k);   // fp32 add (:56)
    double carry = (double)r0p - (double)rad0;
    for (int f0i = 0; f0i < Fb; f0i += 32) {
        const int f = f0i + lane;
        double v = (f < Fb) ? (double)d.U * (double)rad_of(f0b[f], k, d.sr) : 0.0;
        double incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (f < Fb) out[f] = carry + (incl - v);
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// v[t] in double for one sample (needs S1[t], S1[t-1]); also returns rad.
__device__ __forceinline__ double nsf_v(const NsfDims &d, const float *f0b, const double *base1, int k, int t,
                                        float r0p) {
    const int f = t / d.U, j = t - f * d.U;
    const float rad = rad_of(f0b[f], k, d.sr);
    if (t == 0) return (double)r0p;                                // first sample carries the initial phase
    // base1[f] is S1 at the last sample of frame f-1, so S1[t-1] = base1[f] + j * rad for every t > 0
    const double s1 = base1[f] + (double)(j + 1) * (double)rad;
    const double s1m = base1[f] + (double)j * (double)rad;
    const float fr = fmodf((float)s1, 1.0f), frm = fmodf((float)s1m, 1.0f);   // cumsum -> fp32, % 1 (:66)
    const bool wrap = (fr - frm) < 0.f;                                        // (:67-68)
    const float v = wrap ? (rad + -1.0f) : rad;                                // rad + cumsum_shift (:72)
    return (double)v;
}

// ---- kernel 2: per-chunk (32 samples) sums of v, one warp per (b, k, chunk) --------------------
__global__ void nsf_chunk_sum_kernel(NsfDims d, const float *__restrict__ f0, const float *__restrict__ rand_ini,
                                     uint64_t seed, const double *__restrict__ base1, double *__restrict__ csum) {
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= (long long)d.B * kH * d.nchunk) return;
    const int chunk = (int)(wid % d.nchunk);
    const int bk = (int)(wid / d.nchunk), b = bk / kH, k = bk % kH;
    const int Tb = d.frames(b) * d.U;
    if (chunk * 32 >= Tb) {                                   // past the clip: contributes nothing to its scan
        if (lane == 0) csum[wid] = 0.0;
        return;
    }
    const float *f0b = d.f0_of(f0, b);
    const float r0p = rad_of(f0b[0], k, d.sr) + rand_ini_of(rand_ini, seed, b, k);
    const int t = chunk * 32 + lane;
    double v = (t < Tb) ? nsf_v(d, f0b, base1 + (size_t)bk * d.F, k, t, r0p) : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) csum[wid] = v;
}

// ---- kernel 3: exclusive scan of the chunk sums, one warp per (b, k), in place ------------------
__global__ void nsf_chunk_scan_kernel(NsfDims d, double *__restrict__ csum) {
    const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (wid >= d.B * kH) return;
    double *p = csum + (size_t)wid * d.nchunk;
    double carry = 0.0;
    for (int c0 = 0; c0 < d.nchunk; c0 += 32) {
        const int c = c0 + lane;
        const double v = (c < d.nchunk) ? p[c] : 0.0;
        double incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (c < d.nchunk) p[c] = carry + (incl - v);
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
}

// ---- kernel 4: synthesis + harmonic merge, one warp per (b, chunk) -----------------------------
__global__ void nsf_synth_kernel(NsfDims d, const float *__restrict__ f0, const float *__restrict__ rand_ini,
                                 const float *__restrict__ noise, uint64_t seed, const double *__restrict__ base1,
                                 const double *__restrict__ cbase, const float *__restrict__ lin_w, const float *__restrict__ lin_b,
                                 float *__restrict__ har, float *__restrict__ sines) {
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= (long long)d.B * d.nchunk) return;
    const int chunk = (int)(wid % d.nchunk), b = (int)(wid / d.nchunk);
    const int Tb = d.frames(b) * d.U;
    if (chunk * 32 >= Tb) return;                             // past the clip: har there is never read
    const float *f0b = d.f0_of(f0, b);
    const int t = chunk * 32 + lane;
    const bool valid = t < Tb;
    const float f0t = valid ? f0b[t / d.U] : 0.f;
    const float uv = f0t > 0.f ? 1.f : 0.f;                                   // _f02uv (:38-42), threshold 0
    const float noise_amp = uv * 0.003f + (1.f - uv) * 0.1f / 3.f;            // (:131)

    float nz[kH];
    if (noise) {
#pragma unroll
        for (int k = 0; k < kH; ++k) nz[k] = valid ? __ldg(noise + ((size_t)b * d.T + t) * kH + k) : 0.f;
    } else {
        const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const uint4 r = philox4x32_10(make_uint4((uint32_t)t, (uint32_t)b, (uint32_t)g, 0x4e5346u), key);
            float n0, n1, n2, n3;
            box_muller(r.x, r.y, n0, n1);
            box_muller(r.z, r.w, n2, n3);
            nz[3 * g] = n0, nz[3 * g + 1] = n1, nz[3 * g + 2] = n2;
        }
    }

    float merged = __ldg(lin_b);
#pragma unroll 1
    for (int k = 0; k < kH; ++k) {
        const int bk = b * kH + k;
        const float r0p = rad_of(f0b[0], k, d.sr) + rand_ini_of(rand_ini, seed, b, k);
        const double v = valid ? nsf_v(d, f0b, base1 + (size_t)bk * d.F, k, t, r0p) : 0.0;
        double incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        const float s2 = (float)(cbase[(size_t)bk * d.nchunk + chunk] + incl);
        const float sine = sinf(s2 * 2.0f * 3.14159274101257324f) * 0.1f;     // (:72-73,121)
        const float x = sine * uv + noise_amp * nz[k];                         // (:132-136)
        merged = fmaf(__ldg(lin_w + k), x, merged);                            // l_linear (:393)
        if (sines && valid) sines[((size_t)b * d.T + t) * kH + k] = x;         // kept for the l_linear gradient (training)
    }
    if (valid) har[(size_t)b * d.T + t] = tanhf(merged);                       // l_tanh (:394)
}

size_t nsf_workspace_bytes(int B, int F, int U) {
    const size_t T = (size_t)F * U, nchunk = (T + 31) / 32;
    return ((size_t)B * kH * F + (size_t)B * kH * nchunk) * sizeof(double);
}

int launch_nsf_source(const float *f0, const float *rand_ini, const float *noise, uint64_t seed, int B, int F, int U,
                      float sr, const float *lin_w_dev, const float *lin_b_dev, void *workspace, float *har, float *sines,
                      cudaStream_t st, int *launches, const int *len, const int *off) {
    NsfDims d;
    d.B = B, d.F = F, d.U = U, d.T = F * U, d.nchunk = (d.T + 31) / 32, d.sr = sr, d.len = len, d.off = off;
    double *base1 = reinterpret_cast<double *>(workspace);
    double *csum = base1 + (size_t)B * kH * F;
    const int tpb = 128;
    {
        const long long threads = (long long)B * kH * 32;
        nsf_frame_prefix_kernel<<<(unsigned)((threads + tpb - 1) / tpb), tpb, 0, st>>>(d, f0, rand_ini, seed, base1);
    }
    {
        const long long threads = (long long)B * kH * d.nchunk * 32;
        nsf_chunk_sum_kernel<<<(unsigned)((threads + tpb - 1) / tpb), tpb, 0, st>>>(d, f0, rand_ini, seed, base1, csum);
    }
    {
        const long long threads = (long long)B * kH * 32;
        nsf_chunk_scan_kernel<<<(unsigned)((threads + tpb - 1) / tpb), tpb, 0, st>>>(d, csum);
    }
    {
        const long long threads = (long long)B * d.nchunk * 32;
        nsf_synth_kernel<<<(unsigned)((threads + tpb - 1) / tpb), tpb, 0, st>>>(d, f0, rand_ini, noise, seed, base1, csum,
                                                                               lin_w_dev, lin_b_dev, har, sines);
    }
    SVB_CUDA(cudaGetLastError());
    if (launches) *launches += 4;
    return SVB_OK;
}

}  // namespace svb
