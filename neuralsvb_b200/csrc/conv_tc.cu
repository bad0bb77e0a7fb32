// tcgen05 implicit-GEMM 1-D convolution on the G32T activation layout (sm_100a).
//
//   D[128 time rows x N columns] (fp32, TMEM) += A[128 x 16] (bf16, smem) * B[16 x N] (bf16, smem)
//
// GEMM mapping: M = time (128 rows per MMA), N = output channels (<= 128 per CTA), K = taps x Cin.
// * A operand = the activation slab.  G32T keeps, per 32-channel group, consecutive time steps as
//   consecutive 128-byte rows, so the [rows x 32 ch] slab is one contiguous span fetched with ONE
//   cp.async.bulk (TMA, UBLKCP) straight into the operand slot.  The transform warps rewrite it IN
//   PLACE into the MMA operand: leaky-relu pre-activation, hi/lo split (or tf32 rounding) and the
//   SWIZZLE_128B chunk permutation; one 128-byte K-major row per time step.  A conv tap at
//   dilation d is a ROW SHIFT of that operand = +128*k*d bytes on the descriptor start address,
//   so one slab (mt*128 + halo rows) feeds all KS taps of mt accumulator tiles.
// * B operand = weights, packed and pre-swizzled on the host per (column block, input-channel
//   chunk, tap), streamed through a ring of bulk copies (or kept resident for narrow layers).
// * Persistent, warp-specialised: TMA producer warp, MMA warp (TMEM owner; converged-warp issue,
//   see tc_ptx.cuh), 8 operand-transform warps, 8 epilogue warps (tcgen05.ld -> bias / residual /
//   scale / accumulate -> 128-byte row stores) on the accumulator set the MMAs are not writing.
//   HBM tensors stay exact fp32; rounding happens only on the operand copy in smem.
// * One launch runs a WORK LIST: items (layer, column block, clip, first row, tiles) in the order
//   each CTA executes them.  A single layer uses the implicit round-robin list; the generator hands
//   in host-built lists that merge the independent ResBlock chains of a stage into one launch
//   (up to 3 layers of the same shape class, longest-processing-time balanced over the SMs), so the
//   pipeline fill / drain of a persistent launch is paid once per step of the chains, not per layer.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <vector>

#include <cuda_bf16.h>

#include "conv_tc.cuh"
#include "tc_ptx.cuh"

namespace svb {

constexpr int kTcM = 128;       // rows per CTA (UMMA M)
constexpr int kTcCK = 32;       // input channels per chunk = 4 MMAs of K = 8
constexpr int kMaxItems = 120;  // work items per CTA staged in shared memory (16 bytes each)
constexpr int kItemBytes = 2048;


// Operand modes (svb_precision): 1 = 1xTF32, 2 = 3xTF32, 3 = 3xBF16 (hi/lo split, 16-bit mantissa).
// One operand row = 32 input channels = 128 bytes:  TF32: 32 x tf32 ; BF16x3: [32 x bf16 hi | 32 x bf16 lo].
struct TcLayer {                // what differs between the layers of one launch
    const float *in;            // G32T input
    const float *res;           // residual (G32T like out) or nullptr
    float *out;
    const float *bias;
    const unsigned char *w;     // packed, pre-swizzled weight tiles of this layer in the launch's precision mode
    int KS, dil;
    float out_scale;
    int accumulate;
    int bias_off;               // float offset of this layer's bias in the shared-memory bias area
    uint32_t w_res_off;         // resident weights: byte offset of this layer's tiles in the resident area
};

struct TcArgs {
    ConvArgs a;                 // the shape class (B, channels, rows, in_slope, ups_u ...); per-layer fields live in L[]
    TcLayer L[kTcMaxLayers];
    int n_layers;
    const int4 *work;           // explicit work list (device) or nullptr: implicit round-robin over the groups of layer 0
    const int *work_off;        // [grid + 1] item ranges per CTA
    int n_tile, n_chunks, MT, nW, nA, tmem_cols;
    int n_sets;                 // accumulator sets in TMEM: 2 = epilogue of item n overlaps the MMAs of n + 1
    int col_blocks, groups_per_b, total_groups;
    int w_resident;             // every layer's tiles stay in shared memory for the whole launch (narrow layers)
    int blk_chunk_step;         // grouped conv: first input chunk of column block nblk = nblk * blk_chunk_step (0: dense)
    uint32_t w_res_bytes;       // resident: total bytes of all layers' tiles
    int pdl;                    // launched with programmatic stream serialization
    int collect;                // A-operand collector reuse between the two products of a_hi (SVB_TC_COLLECT, default on)
    long long *stats;           // SVB_TC_STATS: [grid][kTcStatSlots] blocked-cycle counters (diagnostics build of the kernel)
    int dbg;                    // SVB_TC_DBG bit mask: 1 no MMAs, 2 hi*hi only, 4 no transform, 8 no epilogue ld/st
    uint32_t op_bytes;          // operand slot: Rp rows x 128 B (x2 with the 3xTF32 lo plane), sized for the largest halo
    uint32_t wtile_bytes;       // one (column block, chunk, tap) weight tile (x2 with the 3xTF32 lo plane)
    uint32_t off_op, off_w, off_stage, off_bias;   // byte offsets of operand slots / weight ring / epilogue tiles / bias in dynamic smem
};

constexpr int kMaxW = 8;
constexpr int kMaxDevices = 64;     // per-device caches of function attributes / SM counts
// Warp roles.  The SM's issue arbiter favours HIGH warp ids, so the two latency-critical single-thread
// roles get the highest ids: warps 0-7 epilogue, 8-15 operand transform, 16 TMA producer, 17 MMA issuer.
constexpr int kTcThreadsP = 576;
constexpr int kWarpProducer = 16, kWarpMma = 17, kWarpTransform0 = 8;
constexpr int kStageBytes = 8 * 4096;   // epilogue transpose tiles: 32 rows x 128 B per epilogue warp
constexpr int kBiasBytes = 4096;        // bias of the layer(s) (<= 1024 floats; wider layers take 12 KB)

// STATS (SVB_TC_STATS=1, diagnostics only): every role accumulates the cycles it spends blocked on each of its
// barriers; the launcher prints the per-CTA mean / max.  Says which stage of the pipeline the others wait for.
template <bool ST>
__device__ __forceinline__ void mbar_wait_t(uint64_t *bar, uint32_t parity, long long &acc) {
    if (ST) {
        const long long t = clock64();
        mbar_wait(bar, parity);
        acc += clock64() - t;
    } else {
        mbar_wait(bar, parity);
    }
}
// wait of a converged single-role warp: every lane polls (measured: one polling lane + __syncwarp for the rest doubles the
// time of every layer), then the warp re-converges -- the uniform-datapath instructions that follow execute once per
// converged warp (tc_ptx.cuh)
template <bool ST>
__device__ __forceinline__ void mbar_wait_warp(uint64_t *bar, uint32_t parity, long long &acc) {
    mbar_wait_t<ST>(bar, parity, acc);
    __syncwarp();
}
constexpr int kTcStatSlots = 16;

// a work item, as staged in shared memory: x = layer | column block << 8 | tiles << 24, y = clip, z = first row,
// w = valid rows of the clip (rows at or past it are not stored; a ragged batch has its own count per clip)
struct TcItem {
    int layer, nblk, mt, b, t0, rows;
};
__device__ __forceinline__ TcItem item_decode(const int4 v) {
    TcItem it;
    it.layer = v.x & 0xff, it.nblk = (v.x >> 8) & 0xffff, it.mt = v.x >> 24, it.b = v.y, it.t0 = v.z, it.rows = v.w;
    return it;
}

// Persistent kernel: one CTA per SM walks its work items (mt consecutive 128-row tiles of one clip for one
// column block of one layer).  Every stage is decoupled by mbarriers, so the TMA producer runs ahead into
// the next item, the transform warps prepare operands while the tensor core works on the previous chunk,
// and the epilogue drains accumulator set (n & 1) from TMEM while the MMAs of item n + 1 fill the other set.
// RG: ragged batch (a.rows != nullptr), the epilogue bounds rows by the item's clip; a separate instantiation keeps the
// uniform kernel's epilogue on the constant a.Tq (one register fewer under the 96-register cap)
template <int MODE, bool ST = false, bool RG = false>
__global__ void __launch_bounds__(kTcThreadsP, 1) conv1d_c4_tc_kernel(const __grid_constant__ TcArgs p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr bool BF = MODE == SVB_PREC_BF16X3;
    constexpr bool X3 = MODE == SVB_PREC_TF32X3;
    const ConvArgs &a = p.a;
    // ---- shared memory carve-up (operand slots and weight ring are 1024-byte aligned: swizzle atoms)
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem);
    uint64_t *raw_full = bars, *a_ready = bars + 4, *a_empty = bars + 8;      // up to 4 operand slots
    uint64_t *w_full = bars + 12, *w_empty = bars + 12 + kMaxW;
    uint64_t *acc_full = bars + 12 + 2 * kMaxW, *acc_empty = acc_full + 2;
    uint32_t *tmem_ptr = reinterpret_cast<uint32_t *>(acc_empty + 2);
    int *n_items_s = reinterpret_cast<int *>(tmem_ptr + 1);
    TcLayer *Ls = reinterpret_cast<TcLayer *>(smem + 512);                    // per-layer table (dynamic indexing)
    const int4 *items = reinterpret_cast<const int4 *>(smem + 1024);         // [kMaxItems]
    unsigned char *op0 = smem + p.off_op;                            // [nA][op_bytes]: TMA target AND MMA operand
    unsigned char *wring = smem + p.off_w;                           // [nW][wtile_bytes] ring, or the resident tiles

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int acc_cols = p.MT * p.n_tile;                            // columns of one accumulator set
    long long st_w0 = 0, st_w1 = 0, st_w2 = 0;                       // STATS: cycles blocked on up to three barriers
    const long long st_t0 = ST ? clock64() : 0;
    unsigned long long st_g0 = 0;
    if (ST) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(st_g0));

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) mbar_init(raw_full + i, 1), mbar_init(a_ready + i, 8), mbar_init(a_empty + i, 1);
        for (int i = 0; i < 2; ++i) mbar_init(acc_full + i, 1), mbar_init(acc_empty + i, 8);
        for (int i = 0; i < kMaxW; ++i) mbar_init(w_full + i, 1), mbar_init(w_empty + i, 1);
        fence_barrier_init();
    }
    if (warp == kWarpMma) tmem_alloc(tmem_ptr, p.tmem_cols);
    {   // constant data (not produced by the previous kernel): staged once, before the PDL wait
        float *sb = reinterpret_cast<float *>(smem + p.off_bias);
        for (int l = 0; l < p.n_layers; ++l)
            for (int i = threadIdx.x; i < a.Cout; i += kTcThreadsP) sb[p.L[l].bias_off + i] = __ldg(p.L[l].bias + i);
        if (threadIdx.x < p.n_layers) Ls[threadIdx.x] = p.L[threadIdx.x];
        int4 *it_w = reinterpret_cast<int4 *>(smem + 1024);
        if (p.work) {                                                // explicit list: this CTA's range
            const int i0 = __ldg(p.work_off + blockIdx.x), n = __ldg(p.work_off + blockIdx.x + 1) - i0;
            for (int i = threadIdx.x; i < n; i += kTcThreadsP) it_w[i] = __ldg(p.work + i0 + i);
            if (threadIdx.x == 0) *n_items_s = n;
        } else if (RG) {                                             // implicit, ragged: only the groups inside each clip
            if (threadIdx.x == 0) {
                int n = 0;
                for (int g = blockIdx.x; g < p.total_groups; g += gridDim.x) {
                    const int tg = g % p.groups_per_b, r = g / p.groups_per_b, b = r % a.B;
                    const int rows = a.rows[b] * a.rows_mul, tiles = (rows + kTcM - 1) / kTcM;
                    if (tg * p.MT >= tiles) continue;
                    it_w[n++] = make_int4(((r / a.B) << 8) | (min(p.MT, tiles - tg * p.MT) << 24), b, tg * (kTcM * p.MT), rows);
                }
                *n_items_s = n;
            }
        } else {                                                     // implicit: groups blockIdx.x, + gridDim.x, ... of layer 0
            const int n = ((int)blockIdx.x < p.total_groups) ? (p.total_groups - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
            for (int i = threadIdx.x; i < n; i += kTcThreadsP) {
                const int g = blockIdx.x + i * gridDim.x;
                const int tg = g % p.groups_per_b, r = g / p.groups_per_b;
                it_w[i] = make_int4(((r / a.B) << 8) | (p.MT << 24), r % a.B, tg * (kTcM * p.MT), a.Tq);
            }
            if (threadIdx.x == 0) *n_items_s = n;
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const int n_items = *n_items_s;
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation) overlapped the
    // tail of the previous kernel in the stream; its results are needed from here on.  The next
    // kernel may begin ITS prologue as soon as every CTA of this grid has reached this point.
    if (p.pdl) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }

    // The two single-warp roles below are latency-critical (every instruction they execute sits
    // between two TMA copies or two MMAs), so all ring indices / phases are kept as incrementing
    // counters -- no runtime integer divisions in the loops.
    if (warp == kWarpProducer) {
        // ================================ TMA producer ================================
        // One bulk copy per slab (rows x 128 B, contiguous in G32T) and one per weight tile, issued by one lane (measured:
        // a converged producer warp is no faster -- the copies are far from their issue limit -- and its item-dependent
        // addresses would have to be made warp-uniform first, see the MMA warp).
        if (lane == 0) {
            const int gin = c4t_groups(a.Cin);
            const size_t group_stride = (size_t)a.in_Tp * 32;                     // floats between channel groups
            int sA = 0, phA = 1, sW = 0, phW = 1;                                 // "empty" barriers start free
            if (p.w_resident && n_items > 0) {                                    // all layers' tiles, once
                mbar_expect_tx(w_full, p.w_res_bytes);
                for (int l = 0; l < p.n_layers; ++l)
                    bulk_g2s(wring + Ls[l].w_res_off, Ls[l].w, (uint32_t)Ls[l].KS * p.wtile_bytes, w_full);
            }
            for (int n = 0; n < n_items; ++n) {
                const TcItem it = item_decode(items[n]);
                const TcLayer &L = Ls[it.layer];
                const int halo = (L.KS - 1) / 2 * L.dil;
                const uint32_t raw_bytes = (uint32_t)(it.mt * kTcM + 2 * halo) * 128;
                const float *in_c = L.in + (((size_t)it.b * gin + (size_t)it.nblk * p.blk_chunk_step) * a.in_Tp + (kPad + it.t0 - halo)) * 32;
                const unsigned char *w_k = L.w + (size_t)it.nblk * p.n_chunks * L.KS * p.wtile_bytes;
                for (int c = 0; c < p.n_chunks; ++c) {
                    mbar_wait_t<ST>(a_empty + sA, phA, st_w0);                    // MMAs of the slot's previous slab retired
                    mbar_expect_tx(raw_full + sA, raw_bytes);
                    bulk_g2s(op0 + sA * p.op_bytes, in_c, raw_bytes, raw_full + sA);
                    in_c += group_stride;
                    if (++sA == p.nA) sA = 0, phA ^= 1;
                    if (!p.w_resident) {
                        for (int k = 0; k < L.KS; ++k) {
                            mbar_wait_t<ST>(w_empty + sW, phW, st_w1);
                            mbar_expect_tx(w_full + sW, p.wtile_bytes);
                            bulk_g2s(wring + sW * p.wtile_bytes, w_k, p.wtile_bytes, w_full + sW);
                            w_k += p.wtile_bytes;
                            if (++sW == p.nW) sW = 0, phW ^= 1;
                        }
                    }
                }
            }
            if (ST) {
                long long *o = p.stats + (size_t)blockIdx.x * kTcStatSlots;
                o[0] = st_w0, o[1] = st_w1, o[2] = clock64() - st_t0;
            }
        }
    } else if (warp == kWarpMma) {
        // ================================ MMA issuer ==================================
        // The whole warp walks the loop CONVERGED and every MMA / commit is predicated on the elected lane, so the
        // descriptors stay in uniform registers (tc_ptx.cuh, "issue discipline": a divergent single-thread issuer
        // costs 65-82 cycles per MMA, more than the MMA itself for every N below 256).
        const uint32_t elected = elect_one_sync();
        const uint32_t idesc = umma_idesc(BF ? 1 : 2, kTcM, p.n_tile);
        const uint32_t hi_word = desc_hi_sw128(0);
        // Descriptors are advanced in their ENCODED form (address >> 4 in the low 14 bits; every offset below is a
        // multiple of 16 bytes and the sum stays inside shared memory, so the field cannot overflow): one uniform
        // add per operand and MMA -- the issue loop, not the tensor pipe, sets the pace of the narrow layers.
        const uint32_t a_lo_plane = (X3 ? p.op_bytes / 2 : 64u) >> 4;      // lo plane / half-row
        const uint32_t b_lo_plane = (X3 ? p.wtile_bytes / 2 : 64u) >> 4;
        const uint32_t op_base = desc_lo(smem_u32(op0)), w_base = desc_lo(smem_u32(wring));
        const uint32_t op_step = p.op_bytes >> 4, wtile_step = p.wtile_bytes >> 4;
        // the ablation switches exist only in the diagnostics instantiation
        const bool mma_on = ST ? !(p.dbg & 1) : true, hh_only = ST ? (p.dbg & 2) != 0 : false, collect = ST ? p.collect != 0 : true;
        int sA = 0, phA = 0, sW = 0, phW = 0, as = 0, phE = 1;
        if (p.w_resident && n_items > 0) {
            mbar_wait_warp<ST>(w_full, 0, st_w2);
            tc_fence_after();
        }
        const int n_items_u = __reduce_max_sync(0xffffffffu, n_items);
        for (int n = 0; n < n_items_u; ++n) {
            // The item comes from shared memory, i.e. in a vector register the compiler must assume divergent: with it
            // every loop bound / descriptor below turns into per-MMA VOTEU / R2UR traffic (+25 % on the narrow layers).
            // A warp reduction (REDUX) hands the same value back in a UNIFORM register; the layer's fields are then
            // read from the kernel parameters (constant bank, uniform index).
            const int ix = __reduce_max_sync(0xffffffffu, items[n].x);
            const int layer = ix & 0xff, mt = ix >> 24;
            const int KS = p.L[layer].KS;
            const uint32_t tap_step = (uint32_t)p.L[layer].dil * (128 >> 4);   // a tap is a row shift of the operand
            const uint32_t w_res_off = p.L[layer].w_res_off >> 4;
            mbar_wait_warp<ST>(acc_empty + as, phE, st_w0);                   // epilogue has drained this accumulator set
            tc_fence_after();
            const uint32_t d_set = tmem_base + (uint32_t)(as * acc_cols);
            uint32_t fresh = 1;                                               // first MMA of the item overwrites
            for (int c = 0; c < p.n_chunks; ++c) {
                mbar_wait_warp<ST>(a_ready + sA, phA, st_w1);
                tc_fence_after();
                uint32_t a_tap = op_base + sA * op_step;
                uint32_t b_tap = w_base + w_res_off;                          // resident tiles (single chunk)
                for (int k = 0; k < KS; ++k) {
                    if (!p.w_resident) {
                        mbar_wait_warp<ST>(w_full + sW, phW, st_w2);
                        tc_fence_after();
                        b_tap = w_base + sW * wtile_step;
                    }
                    if (mma_on) {
                        uint32_t d = d_set, a_row = a_tap;
#pragma unroll 1
                        for (int m = 0; m < mt; ++m) {
                            const uint32_t acc = fresh ^ 1u;
                            if (BF) {                               // 2 x 16 channels; small cross terms first
                                if (hh_only) {
                                    umma<true>(d, a_row, hi_word, b_tap, hi_word, idesc, acc, elected);
                                    umma<true>(d, a_row + 2, hi_word, b_tap + 2, hi_word, idesc, 1u, elected);
                                } else if (collect) {               // a_hi is read from shared memory once for its two products
                                    umma<true>(d, a_row + a_lo_plane, hi_word, b_tap, hi_word, idesc, acc, elected);
                                    umma<true, 1>(d, a_row, hi_word, b_tap + b_lo_plane, hi_word, idesc, 1u, elected);
                                    umma<true, 2>(d, a_row, hi_word, b_tap, hi_word, idesc, 1u, elected);
                                    umma<true>(d, a_row + a_lo_plane + 2, hi_word, b_tap + 2, hi_word, idesc, 1u, elected);
                                    umma<true, 1>(d, a_row + 2, hi_word, b_tap + b_lo_plane + 2, hi_word, idesc, 1u, elected);
                                    umma<true, 2>(d, a_row + 2, hi_word, b_tap + 2, hi_word, idesc, 1u, elected);
                                } else {
                                    umma<true>(d, a_row + a_lo_plane, hi_word, b_tap, hi_word, idesc, acc, elected);
                                    umma<true>(d, a_row, hi_word, b_tap + b_lo_plane, hi_word, idesc, 1u, elected);
                                    umma<true>(d, a_row, hi_word, b_tap, hi_word, idesc, 1u, elected);
                                    umma<true>(d, a_row + a_lo_plane + 2, hi_word, b_tap + 2, hi_word, idesc, 1u, elected);
                                    umma<true>(d, a_row + 2, hi_word, b_tap + b_lo_plane + 2, hi_word, idesc, 1u, elected);
                                    umma<true>(d, a_row + 2, hi_word, b_tap + 2, hi_word, idesc, 1u, elected);
                                }
                            } else {
#pragma unroll
                                for (uint32_t kb = 0; kb < 8; kb += 2) {   // 4 x 8 channels (32 bytes = 2 descriptor units each)
                                    const uint32_t acc_k = kb == 0 ? acc : 1u;
                                    if (X3) {
                                        umma<false>(d, a_row + a_lo_plane + kb, hi_word, b_tap + kb, hi_word, idesc, acc_k, elected);
                                        umma<false, 1>(d, a_row + kb, hi_word, b_tap + b_lo_plane + kb, hi_word, idesc, 1u, elected);
                                        umma<false, 2>(d, a_row + kb, hi_word, b_tap + kb, hi_word, idesc, 1u, elected);
                                    } else {
                                        umma<false>(d, a_row + kb, hi_word, b_tap + kb, hi_word, idesc, acc_k, elected);
                                    }
                                }
                            }
                            d += (uint32_t)p.n_tile, a_row += (kTcM * 128) >> 4;
                        }
                    }
                    fresh = 0;
                    a_tap += tap_step, b_tap += wtile_step;
                    if (!p.w_resident) {                            // tile consumed: release its ring slot
                        umma_commit(w_empty + sW, elected);
                        if (++sW == p.nW) sW = 0, phW ^= 1;
                    }
                }
                umma_commit(a_empty + sA, elected);
                if (++sA == p.nA) sA = 0, phA ^= 1;
            }
            umma_commit(acc_full + as, elected);
            if (++as == p.n_sets) as = 0, phE ^= 1;
        }
        if (ST && elected) {
            long long *o = p.stats + (size_t)blockIdx.x * kTcStatSlots;
            o[3] = st_w0, o[4] = st_w1, o[5] = st_w2, o[6] = clock64() - st_t0;
        }
    } else if (warp >= kWarpTransform0) {
        // ====================== operand transform warps (256 threads) =================
        // In place, 8 lanes per 128-byte row (one 16-byte chunk = 4 channels each): conflict-free
        // LDS.128 / STS.128.  Row r, logical chunk j is stored at chunk position j ^ (r & 7)
        // (SWIZZLE_128B).  bf16 mode: lane pairs exchange halves so the even lane writes the
        // 8-channel hi chunk (j = c/2) and the odd lane the lo chunk (4 + c/2).
        const int tid = threadIdx.x - kWarpTransform0 * 32;     // 0..255
        const int cl = tid & 7;                                 // chunk of the row this lane reads
        const bool odd = cl & 1;
        const float slope = a.in_slope;                         // 0 <= slope <= 1: lrelu(x) = max(x, slope * x)
        int sA = 0, phA = 0;
        for (int n = 0; n < n_items; ++n) {
            const TcItem it = item_decode(items[n]);
            const int R = it.mt * kTcM + (Ls[it.layer].KS - 1) / 2 * Ls[it.layer].dil * 2;
            for (int c = 0; c < p.n_chunks; ++c) {
                mbar_wait_t<ST>(raw_full + sA, phA, st_w0);
                uint4 *op = reinterpret_cast<uint4 *>(op0 + sA * p.op_bytes);
                // 64 rows per pass over the 256 threads: two independent rows per thread for ILP
                for (int r0 = 0; r0 < ((p.dbg & 4) ? 0 : R); r0 += 64) {
                    int rr[2];
                    bool ok[2];
                    float4 v[2];
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        rr[u] = r0 + 32 * u + (tid >> 3);
                        ok[u] = rr[u] < R;
                        v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok[u]) v[u] = *reinterpret_cast<const float4 *>(op + (size_t)rr[u] * 8 + cl);
                    }
#pragma unroll
                    for (int u = 0; u < 2; ++u) {
                        float4 &x = v[u];
                        x.x = fmaxf(x.x, x.x * slope), x.y = fmaxf(x.y, x.y * slope);
                        x.z = fmaxf(x.z, x.z * slope), x.w = fmaxf(x.w, x.w * slope);
                    }
                    if (BF) {
                        uint32_t h0[2], h1[2], l0[2], l1[2], g0[2], g1[2];
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            const __nv_bfloat162 hA = __floats2bfloat162_rn(v[u].x, v[u].y), hB = __floats2bfloat162_rn(v[u].z, v[u].w);
                            h0[u] = *reinterpret_cast<const uint32_t *>(&hA), h1[u] = *reinterpret_cast<const uint32_t *>(&hB);
                            const __nv_bfloat162 lA = __floats2bfloat162_rn(v[u].x - __uint_as_float(h0[u] << 16),
                                                                           v[u].y - __uint_as_float(h0[u] & 0xffff0000u));
                            const __nv_bfloat162 lB = __floats2bfloat162_rn(v[u].z - __uint_as_float(h1[u] << 16),
                                                                           v[u].w - __uint_as_float(h1[u] & 0xffff0000u));
                            l0[u] = *reinterpret_cast<const uint32_t *>(&lA), l1[u] = *reinterpret_cast<const uint32_t *>(&lB);
                        }
                        // even lane keeps hi and receives the neighbour's hi; odd lane keeps lo (shuffles also order reads before writes)
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            g0[u] = __shfl_xor_sync(0xffffffffu, odd ? h0[u] : l0[u], 1);
                            g1[u] = __shfl_xor_sync(0xffffffffu, odd ? h1[u] : l1[u], 1);
                        }
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            if (!ok[u]) continue;
                            uint4 *row = op + (size_t)rr[u] * 8;
                            const int sw = rr[u] & 7;
                            if (!odd) row[(cl >> 1) ^ sw] = make_uint4(h0[u], h1[u], g0[u], g1[u]);          // channels 8j..8j+7 hi
                            else row[(4 + (cl >> 1)) ^ sw] = make_uint4(g0[u], g1[u], l0[u], l1[u]);          // channels 8j..8j+7 lo
                        }
                    } else {
                        __syncwarp();
#pragma unroll
                        for (int u = 0; u < 2; ++u) {
                            if (!ok[u]) continue;
                            uint4 *row = op + (size_t)rr[u] * 8;
                            const int sw = rr[u] & 7;
                            const float4 h = make_float4(to_tf32(v[u].x), to_tf32(v[u].y), to_tf32(v[u].z), to_tf32(v[u].w));
                            row[cl ^ sw] = make_uint4(__float_as_uint(h.x), __float_as_uint(h.y), __float_as_uint(h.z), __float_as_uint(h.w));
                            if (X3)
                                (row + p.op_bytes / 32)[cl ^ sw] =
                                    make_uint4(__float_as_uint(to_tf32(v[u].x - h.x)), __float_as_uint(to_tf32(v[u].y - h.y)),
                                               __float_as_uint(to_tf32(v[u].z - h.z)), __float_as_uint(to_tf32(v[u].w - h.w)));
                        }
                    }
                }
                fence_proxy_async();                                // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(a_ready + sA);           // one arrival per warp (8 per slab)
                if (++sA == p.nA) sA = 0, phA ^= 1;
            }
        }
        if (ST && tid == 0) {
            long long *o = p.stats + (size_t)blockIdx.x * kTcStatSlots;
            o[7] = st_w0, o[8] = clock64() - st_t0;
        }
    } else {
        // ================================ epilogue warps (256 threads) ================
        // TMEM lane = time row, column = output channel; a warp may only touch lanes 32*(warp%4)..+31,
        // so two warps share each lane quarter and alternate over the 32-column blocks.  A block is
        // 32 rows x 128 B, contiguous in G32T.  Global accesses use the "wide" mapping (lane l, step i
        // -> row 4i + l/8, chunk l%8: 512 contiguous bytes per instruction); TMEM hands each thread
        // one whole row, so a per-warp 4 KB swizzled smem tile transposes between the two views.
        // The residual block for step n+1 is requested before block n is drained.
        const int ew = warp;                                        // 0..7
        const int lane_base = 32 * (warp & 3);
        const int half = ew >> 2;                                   // 0 / 1: which blocks this warp takes
        const int gout = c4t_groups(a.Cout);
        float4 *tile = reinterpret_cast<float4 *>(smem + p.off_stage + ew * 4096);   // [32 rows][8 chunks], chunk ^ (row & 7)
        const int jb = p.n_tile / 32;
        const int wr = lane >> 3, wc = lane & 7;                    // wide mapping: row offset / chunk
        const bool no_mem = p.dbg & 8;
        const size_t rstep = (size_t)(a.ups_u > 0 ? a.ups_u : 1) * 8;      // float4 between consecutive GEMM rows
        float4 rres[8];
        // (item, block) -> float4 index of row (q_base + 0) of its 32-row x 128-byte tile; rows are rstep apart;
        // q_base = first GEMM row of this warp in the block
        auto block_base = [&](const TcItem &it, int blk, int &co0, int &q_base) -> size_t {
            const int m = blk / jb, j = blk - m * jb;
            q_base = it.t0 + m * kTcM + lane_base;
            const int cop0 = it.nblk * p.n_tile + j * 32;           // 32 columns never straddle an upsampler phase
            int phi = 0;
            co0 = cop0;
            if (a.ups_u > 0) { phi = cop0 / a.Cout; co0 = cop0 - phi * a.Cout; }
            return (((size_t)it.b * gout + (co0 >> 5)) * a.out_Tp + kPad +
                    (a.ups_u > 0 ? (size_t)q_base * a.ups_u + phi : (size_t)q_base)) * 8;
        };
        // residual rows of one block in the wide mapping -> registers (latency hidden behind the current block)
        auto fetch_res = [&](int n, int blk) {
            if (no_mem || n >= n_items) return;
            const TcItem it = item_decode(items[n]);
            const float4 *res4 = reinterpret_cast<const float4 *>(Ls[it.layer].res);
            if (!res4 || blk >= it.mt * jb) return;
            int co0, q_base;
            const size_t base = block_base(it, blk, co0, q_base);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int rr = 4 * i + wr;
                rres[i] = (q_base + rr < (RG ? it.rows : a.Tq)) ? __ldg(res4 + base + (size_t)rr * rstep + wc) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        fetch_res(0, half);
        int as = 0, phF = 0;
        for (int n = 0; n < n_items; ++n) {
            const TcItem it = item_decode(items[n]);
            const TcLayer &L = Ls[it.layer];
            const bool has_res = L.res != nullptr;
            float4 *out4 = reinterpret_cast<float4 *>(L.out);
            const float out_scale = L.out_scale;
            const int accumulate = L.accumulate;
            const unsigned char *bias_s = smem + p.off_bias + (size_t)L.bias_off * 4;
            const int nblocks = it.mt * jb;
            mbar_wait_t<ST>(acc_full + as, phF, st_w0);
            tc_fence_after();
            for (int blk = half; blk < nblocks; blk += 2) {
                const int m = blk / jb, j = blk - m * jb;
                int co0, q_base;
                const size_t base = block_base(it, blk, co0, q_base);
                if (has_res) {                                       // residual: wide registers -> tile
#pragma unroll
                    for (int i = 0; i < 8; ++i) tile[(4 * i + wr) * 8 + (wc ^ ((4 * i + wr) & 7))] = rres[i];
                    __syncwarp();
                }
                // prefetch the residual of this warp's NEXT block: same item, or the first one of its next item
                if (blk + 2 < nblocks) fetch_res(n, blk + 2);
                else fetch_res(n + 1, half);
                // own row: accumulator + bias (+ residual) -> tile, 16 columns at a time (register budget: 18 warps x 96)
#pragma unroll
                for (int hq = 0; hq < 2; ++hq) {
                    float v[16];
                    tmem_ld16(tmem_base + ((uint32_t)lane_base << 16) + (uint32_t)(as * acc_cols + m * p.n_tile + j * 32 + hq * 16), v);
#pragma unroll
                    for (int g4 = 0; g4 < 4; ++g4) {
                        const int gq = hq * 4 + g4;
                        const float4 bv = *reinterpret_cast<const float4 *>(bias_s + (size_t)(co0 + 4 * gq) * 4);
                        float4 o = make_float4(v[4 * g4] + bv.x, v[4 * g4 + 1] + bv.y, v[4 * g4 + 2] + bv.z, v[4 * g4 + 3] + bv.w);
                        float4 *slot = tile + lane * 8 + (gq ^ (lane & 7));
                        if (has_res) {
                            const float4 rv = *slot;
                            o.x += rv.x, o.y += rv.y, o.z += rv.z, o.w += rv.w;
                        }
                        o.x *= out_scale, o.y *= out_scale, o.z *= out_scale, o.w *= out_scale;
                        *slot = o;
                    }
                }
                __syncwarp();
                // tile -> global, wide mapping (512 contiguous bytes per store instruction)
                if (!no_mem) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int rr = 4 * i + wr;
                        if (q_base + rr >= (RG ? it.rows : a.Tq)) continue;
                        float4 o = tile[rr * 8 + (wc ^ (rr & 7))];
                        float4 *dst = out4 + base + (size_t)rr * rstep + wc;
                        if (accumulate) {                            // same thread wrote *dst in the item before (chain-ordered lists)
                            const float4 old = *dst;
                            o.x += old.x, o.y += old.y, o.z += old.z, o.w += old.w;
                        }
                        *dst = o;
                    }
                }
                __syncwarp();
            }
            if (half >= nblocks) fetch_res(n + 1, half);            // idle on this item (one block): still owes the next item's prefetch
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + as);             // this accumulator set may be overwritten
            if (++as == p.n_sets) as = 0, phF ^= 1;
        }
        if (ST && threadIdx.x == 0) {
            long long *o = p.stats + (size_t)blockIdx.x * kTcStatSlots;
            o[9] = st_w0, o[10] = clock64() - st_t0;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (ST && threadIdx.x == 0) {
        unsigned long long g1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
        p.stats[(size_t)blockIdx.x * kTcStatSlots + 11] = clock64() - st_t0;
        p.stats[(size_t)blockIdx.x * kTcStatSlots + 12] = (long long)st_g0;      // absolute ns: first start / last end over the grid
        p.stats[(size_t)blockIdx.x * kTcStatSlots + 13] = (long long)g1;
    }
    if (warp == kWarpMma) {
        tc_fence_after();
        tmem_dealloc(tmem_base, p.tmem_cols);
    }
}

// ------------------------------------------------------------------ host side
static float host_tf32(float x) {   // round to nearest, ties away (cvt.rna.tf32.f32)
    uint32_t u;
    std::memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return x;
    u += 0x1000u;
    u &= 0xFFFFE000u;
    float r;
    std::memcpy(&r, &u, 4);
    return r;
}
static uint16_t host_bf16(float x) {   // round to nearest even (__float2bfloat16_rn)
    uint32_t u;
    std::memcpy(&u, &x, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
static float bf16_to_float(uint16_t h) {
    const uint32_t u = (uint32_t)h << 16;
    float r;
    std::memcpy(&r, &u, 4);
    return r;
}

static int pick_n_tile(int CoutP) {      // columns per CTA: a multiple of 32 (one G32T channel group per epilogue block)
    if (CoutP % 32 != 0) return 0;
    if (CoutP <= 128) return CoutP;
    for (int n = 128; n >= 32; n -= 32)
        if (CoutP % n == 0) return n;
    return 0;
}

// Weight tiles in K-major SWIZZLE_128B order: row n (output column) = 128 bytes holding the 32 input
// channels of the chunk; the 16-byte chunk c of row n is stored at chunk position c ^ (n & 7).
int tc_pack_weights(const float *packed, int KS, int Cin, int CoutP, TcWeights *out, std::vector<void *> *allocs, int force_n_tile) {
    out->KS = KS, out->Cin = Cin, out->CoutP = CoutP, out->ok = false;
    const int n_tile = force_n_tile > 0 ? force_n_tile : pick_n_tile(CoutP);
    if (force_n_tile > 0 && (CoutP % force_n_tile != 0 || force_n_tile % 32 != 0 || force_n_tile > 128)) return SVB_OK;
    if (n_tile == 0 || n_tile % 8 != 0 || Cin % 4 != 0) return SVB_OK;    // CUDA cores handle it
    out->n_tile = n_tile;
    // input channels are padded to whole 32-channel groups (zero weights against the zero pad channels of G32T)
    const int n_chunks = (Cin + kTcCK - 1) / kTcCK, n_blk = CoutP / n_tile;
    const size_t tile_b = (size_t)n_tile * 128;                    // bytes per tile plane
    const size_t n_tiles = (size_t)n_blk * n_chunks * KS;
    std::vector<unsigned char> tf(n_tiles * tile_b), tf3(n_tiles * tile_b * 2), bf(n_tiles * tile_b);
    for (int nb = 0; nb < n_blk; ++nb)
        for (int c = 0; c < n_chunks; ++c)
            for (int k = 0; k < KS; ++k) {
                const size_t t = ((size_t)nb * n_chunks + c) * KS + k;
                float *t1 = reinterpret_cast<float *>(tf.data() + t * tile_b);
                float *t3h = reinterpret_cast<float *>(tf3.data() + t * tile_b * 2);
                float *t3l = reinterpret_cast<float *>(tf3.data() + t * tile_b * 2 + tile_b);
                uint16_t *tb = reinterpret_cast<uint16_t *>(bf.data() + t * tile_b);
                for (int n = 0; n < n_tile; ++n)
                    for (int ci = 0; ci < kTcCK; ++ci) {
                        const int cin_i = c * kTcCK + ci;
                        const float w = cin_i < Cin ? packed[((size_t)k * Cin + cin_i) * CoutP + nb * n_tile + n] : 0.f;
                        const float h = host_tf32(w);
                        const int c16 = ci >> 2;                   // fp32: 4 channels per 16-byte chunk
                        const size_t i4 = (size_t)n * 32 + ((c16 ^ (n & 7)) << 2) + (ci & 3);
                        t1[i4] = h, t3h[i4] = h, t3l[i4] = host_tf32(w - h);
                        const uint16_t bh = host_bf16(w), bl = host_bf16(w - bf16_to_float(bh));
                        const int ch = ci >> 3, cl = 4 + (ci >> 3); // bf16: 8 channels per chunk; hi chunks 0-3, lo 4-7
                        tb[(size_t)n * 64 + ((ch ^ (n & 7)) << 3) + (ci & 7)] = bh;
                        tb[(size_t)n * 64 + ((cl ^ (n & 7)) << 3) + (ci & 7)] = bl;
                    }
            }
    auto up = [&](const void *src, size_t bytes, void **dst) -> int {
        SVB_CUDA(cudaMalloc(dst, bytes));
        allocs->push_back(*dst);
        SVB_CUDA(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
        return SVB_OK;
    };
    SVB_TRY(up(tf.data(), tf.size(), &out->blob[SVB_PREC_TF32]));
    SVB_TRY(up(tf3.data(), tf3.size(), &out->blob[SVB_PREC_TF32X3]));
    SVB_TRY(up(bf.data(), bf.size(), &out->blob[SVB_PREC_BF16X3]));
    out->ok = true;
    return SVB_OK;
}

// device twin of the loops in tc_pack_weights: one thread per (tile, output column n, input channel ci)
__global__ void tc_repack_kernel(const float *__restrict__ packed, int KS, int Cin, int CoutP, int n_tile, int n_chunks,
                                 long long total, unsigned char *__restrict__ tf, unsigned char *__restrict__ tf3,
                                 unsigned char *__restrict__ bf) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int ci = (int)(i % kTcCK);
    const int n = (int)((i / kTcCK) % n_tile);
    const long long t = i / ((long long)kTcCK * n_tile);
    const int k = (int)(t % KS);
    const int c = (int)((t / KS) % n_chunks);
    const int nb = (int)(t / ((long long)KS * n_chunks));
    const int cin_i = c * kTcCK + ci;
    const float w = cin_i < Cin ? packed[((size_t)k * Cin + cin_i) * CoutP + nb * n_tile + n] : 0.f;
    auto tf32 = [](float x) {      // host_tf32: round half up in magnitude to 10 mantissa bits
        uint32_t u = __float_as_uint(x);
        if ((u & 0x7F800000u) == 0x7F800000u) return x;
        u += 0x1000u;
        u &= 0xFFFFE000u;
        return __uint_as_float(u);
    };
    const size_t tile_b = (size_t)n_tile * 128;
    const float h = tf32(w);
    const size_t i4 = (size_t)n * 32 + (((ci >> 2) ^ (n & 7)) << 2) + (ci & 3);
    reinterpret_cast<float *>(tf + t * tile_b)[i4] = h;
    reinterpret_cast<float *>(tf3 + t * tile_b * 2)[i4] = h;
    reinterpret_cast<float *>(tf3 + t * tile_b * 2 + tile_b)[i4] = tf32(w - h);
    const __nv_bfloat16 bh = __float2bfloat16_rn(w);
    const __nv_bfloat16 bl = __float2bfloat16_rn(w - __bfloat162float(bh));
    uint16_t *tb = reinterpret_cast<uint16_t *>(bf + t * tile_b);
    const int ch = ci >> 3, cl = 4 + (ci >> 3);
    tb[(size_t)n * 64 + ((ch ^ (n & 7)) << 3) + (ci & 7)] = __bfloat16_as_ushort(bh);
    tb[(size_t)n * 64 + ((cl ^ (n & 7)) << 3) + (ci & 7)] = __bfloat16_as_ushort(bl);
}

int tc_repack_weights_dev(const float *packed_dev, const TcWeights &w, cudaStream_t st) {
    if (!w.ok) return SVB_OK;
    const int n_chunks = (w.Cin + kTcCK - 1) / kTcCK, n_blk = w.CoutP / w.n_tile;
    const long long total = (long long)n_blk * n_chunks * w.KS * w.n_tile * kTcCK;
    tc_repack_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(
        packed_dev, w.KS, w.Cin, w.CoutP, w.n_tile, n_chunks, total, reinterpret_cast<unsigned char *>(w.blob[SVB_PREC_TF32]),
        reinterpret_cast<unsigned char *>(w.blob[SVB_PREC_TF32X3]), reinterpret_cast<unsigned char *>(w.blob[SVB_PREC_BF16X3]));
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}

bool tc_supported(const TcWeights &w, const ConvArgs &a) {
    if (a.cin_blk > 0 && (a.cin_blk % 32 != 0 || a.ups_u != 0 || (a.CoutP / w.n_tile) * a.cin_blk != a.Cin || w.Cin != a.cin_blk)) return false;
    return w.ok && a.Cin % 4 == 0 && a.bias != nullptr && (a.KS - 1) / 2 * a.dil <= kPad &&
           (a.ups_u == 0 || a.Cout % 32 == 0) && a.Cout <= 3072;
}

template <int MODE, bool ST, bool RG = false>
static int launch_mode(const TcArgs &p, int grid, size_t smem, cudaStream_t st) {
    auto kern = conv1d_c4_tc_kernel<MODE, ST, RG>;
    // function attributes are per device: one process may drive several GPUs (the reference's mp.spawn gives one each,
    // but nothing in the C ABI forbids a handle per device in one process)
    static size_t configured[kMaxDevices] = {};
    static bool carve[kMaxDevices] = {};
    int dev = 0;
    SVB_CUDA(cudaGetDevice(&dev));
    dev = dev < kMaxDevices ? dev : kMaxDevices - 1;
    if (smem > configured[dev] || dev == kMaxDevices - 1) {
        SVB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[dev] = smem;
    }
    if (!carve[dev]) {   // keep the SM's smem/L1 split fixed across the differently-sized launches of a forward
        SVB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        carve[dev] = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid), cfg.blockDim = dim3(kTcThreadsP), cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = p.pdl ? 1 : 0;
    cfg.attrs = attr, cfg.numAttrs = 1;
    SVB_CUDA(cudaLaunchKernelEx(&cfg, kern, p));
    return SVB_OK;
}

static int sm_count() {
    static int n[kMaxDevices] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    const int slot = dev < kMaxDevices ? dev : kMaxDevices - 1;
    if (n[slot] == 0 || slot == kMaxDevices - 1) {
        cudaDeviceGetAttribute(&n[slot], cudaDevAttrMultiProcessorCount, dev);
        if (n[slot] <= 0) n[slot] = 148;
    }
    return n[slot];
}

// Shape-class plan of one launch: M tiles per item, operand slots, weight ring / residency, TMEM columns and the
// shared-memory carve-up.  `a[0..n)` are layers of the same shape class (channels, rows, upsampling) that may
// differ in taps / dilation / pointers; slots are sized for the largest halo.
static int tc_plan(int n, const TcWeights *const *w, const ConvArgs *a, int precision, TcArgs &p, size_t &smem) {
    SVB_CHECK(n >= 1 && n <= kTcMaxLayers, SVB_ERR_INVALID, "tc conv: %d layers in one launch", n);
    const ConvArgs &a0 = a[0];
    for (int l = 1; l < n; ++l)
        SVB_CHECK(a[l].B == a0.B && a[l].Cin == a0.Cin && a[l].Cout == a0.Cout && a[l].CoutP == a0.CoutP && a[l].Tq == a0.Tq &&
                      a[l].in_Tp == a0.in_Tp && a[l].out_Tp == a0.out_Tp && a[l].ups_u == a0.ups_u && a[l].in_slope == a0.in_slope &&
                      a[l].cin_blk == a0.cin_blk && w[l]->n_tile == w[0]->n_tile,
                  SVB_ERR_INVALID, "tc conv: layers of one launch must share the shape class");
    p.a = a0, p.n_layers = n;
    p.work = nullptr, p.work_off = nullptr;
    const int cin_eff = a0.cin_blk > 0 ? a0.cin_blk : a0.Cin;     // input channels one column block contracts over
    p.n_tile = w[0]->n_tile, p.n_chunks = (cin_eff + kTcCK - 1) / kTcCK;
    p.blk_chunk_step = a0.cin_blk > 0 ? p.n_chunks : 0;
    int halo = 0, ks_sum = 0;
    for (int l = 0; l < n; ++l) halo = std::max(halo, (a[l].KS - 1) / 2 * a[l].dil), ks_sum += a[l].KS;
    const int tiles = (a0.Tq + kTcM - 1) / kTcM;              // 128-row tiles per clip
    p.col_blocks = a0.CoutP / p.n_tile;
    const int planes = precision == SVB_PREC_TF32X3 ? 2 : 1;
    p.wtile_bytes = (uint32_t)p.n_tile * 128 * planes;
    p.dbg = 0;
    if (const char *e = getenv("SVB_TC_DBG")) p.dbg = atoi(e);
    p.collect = 1;
    if (const char *e = getenv("SVB_TC_COLLECT")) p.collect = atoi(e) != 0;
    p.pdl = 1;
    if (const char *e = getenv("SVB_TC_PDL")) p.pdl = atoi(e) != 0;
    int force_mt = 0;
    if (const char *e = getenv("SVB_TC_MT")) force_mt = atoi(e);
    // ---- M tiles per item: each weight tile fetched from L2 feeds MT accumulators.  Two accumulator
    // sets live in TMEM (2 * MT * N <= 512 columns); slabs and the weight ring must fit shared memory.
    smem = 0;
    const size_t bias_bytes = (size_t)n * a0.Cout <= 1024 ? kBiasBytes : 3 * kBiasBytes;
    SVB_CHECK((size_t)n * a0.Cout * 4 <= bias_bytes, SVB_ERR_INVALID, "tc conv: %d layers x %d biases exceed the shared-memory bias area", n, a0.Cout);
    const size_t budget = 226 * 1024 - kStageBytes - bias_bytes;
    int force_sets = 0;
    if (const char *e = getenv("SVB_TC_SETS")) force_sets = atoi(e);
    bool planned = false;
    for (int MT : {4, 2, 1}) {
        if (force_mt && MT != force_mt && MT != 1) continue;
        int sets = 2 * MT * p.n_tile <= 512 ? 2 : 1;
        if (force_sets) sets = force_sets;
        if (sets * MT * p.n_tile > 512) continue;
        if (!force_mt) {
            if (MT == 4) continue;      // measured: MT = 4 (one or two accumulator sets) is slower than MT = 2 on every layer
            if (MT == 2 && tiles < 2) continue;
        }
        p.n_sets = sets;
        if ((tiles + MT - 1) / MT * MT * kTcM > round_up(a0.Tq, kTileT) && MT != 1) continue;   // stay inside the allocation
        p.MT = MT;
        const int R = MT * kTcM + 2 * halo;
        p.op_bytes = (uint32_t)round_up(R, 8) * 128 * planes;
        // operand slots double as TMA targets: 3 of them keep two slab copies in flight behind the MMAs
        p.nA = 3;
        if (const char *e = getenv("SVB_TC_NA")) p.nA = std::max(2, std::min(4, atoi(e)));
        p.off_op = 1024 + kItemBytes;
        // narrow layers (one chunk, one column block): every layer's tiles stay resident
        const size_t res_bytes = (size_t)ks_sum * p.wtile_bytes;
        const bool can_res = p.n_chunks == 1 && p.col_blocks == 1;
        p.w_resident = 0;
        for (int nA : {p.nA, 2}) {
            if (can_res && p.off_op + (size_t)nA * p.op_bytes + res_bytes <= budget) {
                p.nA = nA, p.w_resident = 1;
                break;
            }
        }
        p.off_w = p.off_op + (uint32_t)p.nA * p.op_bytes;
        if (!p.w_resident && p.off_w + 2 * (size_t)p.wtile_bytes > budget) {
            p.nA = 2;
            p.off_w = p.off_op + (uint32_t)p.nA * p.op_bytes;
        }
        if (!p.w_resident && p.off_w + 2 * (size_t)p.wtile_bytes > budget && MT != 1) continue;
        SVB_CHECK(p.w_resident || p.off_w + (size_t)p.wtile_bytes <= budget, SVB_ERR_INVALID,
                  "tc conv: tile does not fit shared memory (N %d)", p.n_tile);
        const size_t avail = budget - p.off_w;
        size_t w_area;
        if (p.w_resident) {
            p.nW = 1, p.w_res_bytes = (uint32_t)res_bytes, w_area = res_bytes;
        } else {
            p.nW = std::max(1, std::min((int)(avail / p.wtile_bytes), kMaxW));
            p.w_res_bytes = 0, w_area = (size_t)p.nW * p.wtile_bytes;
        }
        p.off_stage = p.off_w + (uint32_t)round_up((int)w_area, 1024);
        p.off_bias = p.off_stage + kStageBytes;
        smem = (size_t)p.off_bias + bias_bytes;
        planned = true;
        break;
    }
    SVB_CHECK(planned && smem <= 227 * 1024, SVB_ERR_INVALID, "tc conv: no tiling fits (N %d, %d layers)", p.n_tile, n);
    uint32_t res_off = 0;
    for (int l = 0; l < n; ++l) {
        TcLayer &L = p.L[l];
        L.in = a[l].in, L.res = a[l].res, L.out = a[l].out, L.bias = a[l].bias;
        L.w = reinterpret_cast<const unsigned char *>(w[l]->blob[precision]);
        L.KS = a[l].KS, L.dil = a[l].dil, L.out_scale = a[l].out_scale, L.accumulate = a[l].accumulate;
        L.bias_off = l * a0.Cout, L.w_res_off = res_off;
        res_off += (uint32_t)a[l].KS * p.wtile_bytes;
    }
    for (int l = n; l < kTcMaxLayers; ++l) p.L[l] = p.L[0];
    if (getenv("SVB_TC_VERBOSE"))
        fprintf(stderr, "[tc] %d layer(s) Cin %d CoutP %d KS %d.. halo %d Tq %d | n_tile %d MT %d sets %d nA %d nW %d resident %d smem %zu\n", n,
                a0.Cin, a0.CoutP, a0.KS, halo, a0.Tq, p.n_tile, p.MT, p.n_sets, p.nA, p.nW, p.w_resident, smem);
    int cols = 32;
    while (cols < p.n_sets * p.MT * p.n_tile) cols <<= 1;
    p.tmem_cols = cols;
    p.groups_per_b = (tiles + p.MT - 1) / p.MT;
    p.total_groups = p.groups_per_b * a0.B * p.col_blocks;
    p.stats = nullptr;
    return SVB_OK;
}

static int tc_dispatch(TcArgs &p, int precision, int grid, size_t smem, cudaStream_t st) {
    const ConvArgs &a = p.a;
    const bool want_stats = getenv("SVB_TC_STATS") != nullptr;
    if (a.rows) {                                                    // ragged batch
        switch (precision) {
            case SVB_PREC_TF32: return launch_mode<SVB_PREC_TF32, false, true>(p, grid, smem, st);
            case SVB_PREC_TF32X3: return launch_mode<SVB_PREC_TF32X3, false, true>(p, grid, smem, st);
            default: return launch_mode<SVB_PREC_BF16X3, false, true>(p, grid, smem, st);
        }
    }
    if ((want_stats || p.dbg != 0 || !p.collect) && precision == SVB_PREC_BF16X3) {
        // diagnostics: run the instrumented instantiation, wait for it and print where each role was blocked
        const size_t n = (size_t)grid * kTcStatSlots;
        SVB_CUDA(cudaMalloc((void **)&p.stats, n * sizeof(long long)));
        SVB_CUDA(cudaMemsetAsync(p.stats, 0, n * sizeof(long long), st));
        SVB_TRY((launch_mode<SVB_PREC_BF16X3, true>(p, grid, smem, st)));
        SVB_CUDA(cudaStreamSynchronize(st));
        std::vector<long long> h(n);
        SVB_CUDA(cudaMemcpy(h.data(), p.stats, n * sizeof(long long), cudaMemcpyDeviceToHost));
        SVB_CUDA(cudaFree(p.stats));
        double mean[kTcStatSlots] = {};
        long long mx[kTcStatSlots] = {};
        for (int c = 0; c < grid; ++c)
            for (int i = 0; i < kTcStatSlots; ++i) mean[i] += (double)h[(size_t)c * kTcStatSlots + i] / grid, mx[i] = std::max(mx[i], h[(size_t)c * kTcStatSlots + i]);
        long long g_first = h[12], g_last = h[13];
        for (int c = 0; c < grid; ++c) g_first = std::min(g_first, h[(size_t)c * kTcStatSlots + 12]), g_last = std::max(g_last, h[(size_t)c * kTcStatSlots + 13]);
        if (want_stats) fprintf(stderr, "[tc-stats] grid span %.1f us (globaltimer, first CTA start -> last CTA end) = %.2f GHz over the mean CTA\n",
                                (g_last - g_first) / 1e3, mean[11] / std::max(1.0, (double)(g_last - g_first)));
        if (want_stats) fprintf(stderr,
                "[tc-stats] %dx C%d>%d k%d d%d Tq %d grid %d groups %d MT %d | kcycles mean (max): total %.0f (%.0f) | producer: a_empty %.0f w_empty %.0f of %.0f | "
                "mma: acc_empty %.0f a_ready %.0f w_full %.0f of %.0f | transform: raw_full %.0f of %.0f | epilogue: acc_full %.0f of %.0f\n",
                p.n_layers, a.Cin, a.CoutP, a.KS, a.dil, a.Tq, grid, p.total_groups, p.MT, mean[11] / 1e3, mx[11] / 1e3, mean[0] / 1e3, mean[1] / 1e3, mean[2] / 1e3,
                mean[3] / 1e3, mean[4] / 1e3, mean[5] / 1e3, mean[6] / 1e3, mean[7] / 1e3, mean[8] / 1e3, mean[9] / 1e3, mean[10] / 1e3);
        return SVB_OK;
    }
    switch (precision) {
        case SVB_PREC_TF32: return launch_mode<SVB_PREC_TF32, false>(p, grid, smem, st);
        case SVB_PREC_TF32X3: return launch_mode<SVB_PREC_TF32X3, false>(p, grid, smem, st);
        default: return launch_mode<SVB_PREC_BF16X3, false>(p, grid, smem, st);
    }
}

int launch_conv_tc(const TcWeights &w, const ConvArgs &a, int precision, cudaStream_t st, int max_ctas) {
    SVB_CHECK(precision >= SVB_PREC_TF32 && precision <= SVB_PREC_BF16X3, SVB_ERR_INVALID, "tc conv: bad precision %d",
              precision);
    TcArgs p;
    size_t smem = 0;
    const TcWeights *wp = &w;
    SVB_TRY(tc_plan(1, &wp, &a, precision, p, smem));
    const int grid = std::min(p.total_groups, max_ctas > 0 ? std::min(max_ctas, sm_count()) : sm_count());
    if ((p.total_groups + grid - 1) / grid > kMaxItems) {
        // more items per CTA than the shared-memory list holds: run the batch in slices of clips
        const int per_b = p.groups_per_b * p.col_blocks;
        const int nb = std::max(1, kMaxItems * grid / per_b);
        SVB_CHECK(per_b <= kMaxItems * grid, SVB_ERR_INVALID, "tc conv: one clip alone has %d work items", per_b);
        for (int b0 = 0; b0 < a.B; b0 += nb) {
            ConvArgs s = a;
            s.B = std::min(nb, a.B - b0);
            s.in = a.in + (size_t)b0 * c4t_groups(a.Cin) * a.in_Tp * 32;
            s.out = a.out + (size_t)b0 * c4t_groups(a.Cout) * a.out_Tp * 32;
            if (a.res) s.res = a.res + (size_t)b0 * c4t_groups(a.Cout) * a.out_Tp * 32;
            if (a.rows) s.rows = a.rows + b0;
            SVB_TRY(launch_conv_tc(w, s, precision, st, max_ctas));
        }
        return SVB_OK;
    }
    return tc_dispatch(p, precision, grid, smem, st);
}

// whether `n` layers of this shape class fit one merged launch: the per-CTA item list lives in shared memory
bool tc_merge_fits(int n, int B, int Tq, int Cout, int n_tile, const int *rows) {
    long long groups = 0;
    for (int b = 0; b < B; ++b) {
        const int tiles = ((rows ? rows[b] : Tq) + kTcM - 1) / kTcM;
        groups += (tiles + 1) / 2;
    }
    groups *= std::max(1, Cout / std::max(1, n_tile));
    return groups * n <= (long long)(kMaxItems * 8 / 10) * sm_count();
}

// ---- merged launches: several layers of one shape class, host-built balanced work list
void tc_worklist_free(TcWorkList *wl) {
    if (wl->items) cudaFree(wl->items);
    if (wl->off) cudaFree(wl->off);
    *wl = TcWorkList();
}

// The schedule itself is plain host code (no CUDA call): exposed for the CPU tests through svb_tc_schedule_probe.
int tc_schedule(int n, const int *KS, const int *has_res, const int *accum, int Cin, int B, int Tq, int MT, int col_blocks, bool chain_ordered,
                int grid, std::vector<int4> *items_out, std::vector<int> *off_out, double *balance_out, const int *rows) {
    // cost of an item in "taps of one tile": the MMA work plus a constant for the memory-bound part (slab, epilogue)
    const double beta = 160.0 / std::max(32, Cin);
    struct Unit {
        double cost;
        int nblk, b, t0, mt, layer;     // layer < 0: all layers in order (chain-ordered unit)
    };
    auto unit_cost = [&](int layer, int mt) {
        if (layer >= 0) return mt * (KS[layer] + beta + (has_res[layer] ? 1.0 : 0.0));
        double c = 0;
        for (int l = 0; l < n; ++l) c += mt * (KS[l] + beta + (has_res[l] ? 1.0 : 0.0) + (accum[l] ? 1.0 : 0.0));
        return c;
    };
    std::vector<Unit> units;
    for (int nblk = 0; nblk < col_blocks; ++nblk)
        for (int b = 0; b < B; ++b) {
            const int tiles = ((rows ? rows[b] : Tq) + kTcM - 1) / kTcM;       // a ragged clip: its own tile count
            for (int t = 0; t < tiles; t += MT) {
                const int mt = std::min(MT, tiles - t);
                if (chain_ordered) {
                    units.push_back({unit_cost(-1, mt), nblk, b, t * kTcM, mt, -1});
                } else {
                    for (int l = 0; l < n; ++l) units.push_back({unit_cost(l, mt), nblk, b, t * kTcM, mt, l});
                }
            }
        }
    // longest processing time first onto the least-loaded CTA.  Experiment kept behind SVB_TC_SPLIT=1: when the units are
    // too coarse for the 148 SMs (a few per CTA), split the cheapest two-tile units into one-tile halves and redo the
    // schedule.  Measured (same box): nominal balance 0.865 -> 0.95-0.99 but the forward gets 2 % SLOWER (4.66 -> 4.75 ms):
    // a one-tile item streams every weight tile for half the rows.
    std::vector<double> load;
    std::vector<std::vector<int>> mine;
    double balance = 0;
    for (int round = 0; round < 4; ++round) {
        std::stable_sort(units.begin(), units.end(), [](const Unit &x, const Unit &y) { return x.cost > y.cost; });
        load.assign(grid, 0.0);
        mine.assign(grid, std::vector<int>());
        for (size_t u = 0; u < units.size(); ++u) {
            int best = 0;
            for (int c = 1; c < grid; ++c)
                if (load[c] < load[best]) best = c;
            load[best] += units[u].cost;
            mine[best].push_back((int)u);
        }
        double mx = 0, sum = 0;
        for (double v : load) mx = std::max(mx, v), sum += v;
        balance = sum / grid / mx;
        if (balance >= 0.95 || !getenv("SVB_TC_SPLIT")) break;
        // split up to `grid` of the cheapest two-tile units (they sit at the end of the sorted list)
        int split = 0;
        for (size_t u = units.size(); u-- > 0 && split < grid;) {
            if (units[u].mt != 2) continue;
            Unit h0 = units[u], h1 = units[u];
            h0.mt = h1.mt = 1, h1.t0 += kTcM;
            h0.cost = h1.cost = unit_cost(h0.layer, 1);
            units[u] = h0;
            units.push_back(h1);
            ++split;
        }
        if (!split) break;
    }
    std::vector<int4> &items = *items_out;
    std::vector<int> &off = *off_out;
    items.clear();
    off.assign(grid + 1, 0);
    for (int c = 0; c < grid; ++c) {
        // neighbours in time next to each other (their halos share L2 lines)
        std::sort(mine[c].begin(), mine[c].end(), [&](int x, int y) {
            const Unit &X = units[x], &Y = units[y];
            if (X.layer != Y.layer) return X.layer < Y.layer;
            if (X.nblk != Y.nblk) return X.nblk < Y.nblk;
            if (X.b != Y.b) return X.b < Y.b;
            return X.t0 < Y.t0;
        });
        const char *il = getenv("SVB_TC_INTERLEAVE");
        if (!chain_ordered && n > 1 && !(il && atoi(il) == 0)) {
            // alternate the layers inside a CTA (long and short items interleaved) instead of layer after layer: the slab
            // prefetch of a short-kernel item hides behind the MMAs of a long one (measured: 4.67 -> 4.62 ms per forward)
            std::vector<std::vector<int>> by(n);
            for (int u : mine[c]) by[units[u].layer].push_back(u);
            std::vector<int> order;
            std::vector<size_t> pos(n, 0);
            const size_t total = mine[c].size();
            while (order.size() < total) {
                // take from the layer that is furthest behind its proportional share
                int best = -1;
                double lag = -1e30;
                for (int l = 0; l < n; ++l) {
                    if (pos[l] >= by[l].size()) continue;
                    const double want = (double)(order.size() + 1) * by[l].size() / total - (double)pos[l];
                    if (want > lag) lag = want, best = l;
                }
                order.push_back(by[best][pos[best]++]);
            }
            mine[c] = order;
        }
        for (int u : mine[c]) {
            const Unit &U = units[u];
            for (int l = (U.layer < 0 ? 0 : U.layer); l < (U.layer < 0 ? n : U.layer + 1); ++l)
                items.push_back(make_int4(l | (U.nblk << 8) | (U.mt << 24), U.b, U.t0, rows ? rows[U.b] : Tq));
        }
        off[c + 1] = (int)items.size();
        SVB_CHECK(off[c + 1] - off[c] <= kMaxItems, SVB_ERR_INVALID, "tc conv: %d work items on one CTA (limit %d)", off[c + 1] - off[c], kMaxItems);
    }
    *balance_out = balance;
    return SVB_OK;
}

int tc_worklist_build(int n, const TcWeights *const *w, const ConvArgs *a, int precision, bool chain_ordered, TcWorkList *out,
                      const int *rows, cudaStream_t st) {
    TcArgs p;
    size_t smem = 0;
    SVB_TRY(tc_plan(n, w, a, precision, p, smem));
    const int grid = sm_count();
    int KS[kTcMaxLayers], has_res[kTcMaxLayers], accum[kTcMaxLayers];
    for (int l = 0; l < n; ++l) KS[l] = a[l].KS, has_res[l] = a[l].res != nullptr, accum[l] = a[l].accumulate;
    std::vector<int4> items;
    std::vector<int> off;
    double balance = 0;
    SVB_TRY(tc_schedule(n, KS, has_res, accum, a[0].Cin, a[0].B, a[0].Tq, p.MT, p.col_blocks, chain_ordered, grid, &items, &off, &balance,
                        rows));
    // grow-only device buffers, stream-ordered upload: a ragged batch rebuilds its lists on every call with new lengths,
    // and cudaFree would synchronise the device each time
    if (items.size() > out->cap_items || off.size() > out->cap_off) {
        if (out->items) SVB_CUDA(cudaFree(out->items));
        if (out->off) SVB_CUDA(cudaFree(out->off));
        out->items = nullptr, out->off = nullptr;
        out->cap_items = std::max<size_t>(items.size(), 1) * 5 / 4, out->cap_off = off.size();
        SVB_CUDA(cudaMalloc((void **)&out->items, out->cap_items * sizeof(int4)));
        SVB_CUDA(cudaMalloc((void **)&out->off, out->cap_off * sizeof(int)));
    }
    // from pageable memory: the runtime stages the bytes before returning, so the vectors may go out of scope
    SVB_CUDA(cudaMemcpyAsync(out->items, items.data(), items.size() * sizeof(int4), cudaMemcpyHostToDevice, st));
    SVB_CUDA(cudaMemcpyAsync(out->off, off.data(), off.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    out->grid = grid, out->n_items = (int)items.size(), out->MT = p.MT, out->n_layers = n, out->chain_ordered = chain_ordered;
    out->valid = true;
    if (getenv("SVB_TC_VERBOSE"))
        fprintf(stderr, "[tc] work list: %d layers, %zu items over %d CTAs, balance %.3f (mean / max load)\n", n, items.size(), grid, balance);
    return SVB_OK;
}

int launch_conv_tc_multi(int n, const TcWeights *const *w, const ConvArgs *a, int precision, cudaStream_t st, const TcWorkList &wl) {
    SVB_CHECK(precision >= SVB_PREC_TF32 && precision <= SVB_PREC_BF16X3, SVB_ERR_INVALID, "tc conv: bad precision %d", precision);
    TcArgs p;
    size_t smem = 0;
    SVB_TRY(tc_plan(n, w, a, precision, p, smem));
    SVB_CHECK(wl.valid && wl.n_layers == n && wl.MT == p.MT && wl.grid == sm_count(), SVB_ERR_STATE,
              "tc conv: work list was built for another plan (layers %d / %d, MT %d / %d)", wl.n_layers, n, wl.MT, p.MT);
    p.work = wl.items, p.work_off = wl.off;
    return tc_dispatch(p, precision, wl.grid, smem, st);
}

}  // namespace svb

// Host-only view of the merged-launch schedule (no CUDA call): used by the CPU tests to check that every (layer, tile) is
// scheduled exactly once, that chain-ordered lists keep the layers of a tile together and in order, and the LPT balance.
extern "C" int64_t svb_tc_schedule_probe(int32_t n_layers, const int32_t *KS, const int32_t *has_res, const int32_t *accumulate, int32_t Cin,
                                         int32_t B, int32_t Tq, int32_t MT, int32_t col_blocks, int32_t chain_ordered, int32_t grid,
                                         int32_t *items_out, int64_t items_capacity, int32_t *off_out, double *balance_out) {
    SVB_CHECK(n_layers >= 1 && n_layers <= svb::kTcMaxLayers && KS && has_res && accumulate && B > 0 && Tq > 0 && (MT == 1 || MT == 2) &&
                  col_blocks >= 1 && grid >= 1 && items_out && off_out && balance_out,
              SVB_ERR_INVALID, "tc_schedule_probe: bad argument");
    std::vector<int4> items;
    std::vector<int> off;
    int ks[svb::kTcMaxLayers], hr[svb::kTcMaxLayers], ac[svb::kTcMaxLayers];
    for (int l = 0; l < n_layers; ++l) ks[l] = KS[l], hr[l] = has_res[l], ac[l] = accumulate[l];
    SVB_TRY(svb::tc_schedule(n_layers, ks, hr, ac, Cin, B, Tq, MT, col_blocks, chain_ordered != 0, grid, &items, &off, balance_out, nullptr));
    SVB_CHECK((int64_t)items.size() <= items_capacity, SVB_ERR_INVALID, "tc_schedule_probe: %zu items, capacity %lld", items.size(),
              (long long)items_capacity);
    for (size_t i = 0; i < items.size(); ++i) {
        int32_t *o = items_out + 5 * i;                             // layer, column block, clip, first row, tiles
        o[0] = items[i].x & 0xff, o[1] = (items[i].x >> 8) & 0xffff, o[2] = items[i].y, o[3] = items[i].z, o[4] = items[i].x >> 24;
    }
    for (int c = 0; c <= grid; ++c) off_out[c] = off[c];
    return (int64_t)items.size();
}

// The same view for a ragged batch: clip b has rows_per_clip[b] rows (1 <= rows <= Tq).
extern "C" int64_t svb_tc_schedule_probe_ragged(int32_t n_layers, const int32_t *KS, const int32_t *has_res, const int32_t *accumulate,
                                                int32_t Cin, int32_t B, const int32_t *rows_per_clip, int32_t MT, int32_t col_blocks,
                                                int32_t chain_ordered, int32_t grid, int32_t *items_out, int64_t items_capacity,
                                                int32_t *off_out, double *balance_out) {
    SVB_CHECK(n_layers >= 1 && n_layers <= svb::kTcMaxLayers && KS && has_res && accumulate && B > 0 && rows_per_clip && (MT == 1 || MT == 2) &&
                  col_blocks >= 1 && grid >= 1 && items_out && off_out && balance_out,
              SVB_ERR_INVALID, "tc_schedule_probe_ragged: bad argument");
    int Tq = 0;
    for (int b = 0; b < B; ++b) {
        SVB_CHECK(rows_per_clip[b] >= 1, SVB_ERR_INVALID, "tc_schedule_probe_ragged: clip %d has %d rows", b, rows_per_clip[b]);
        Tq = std::max(Tq, (int)rows_per_clip[b]);
    }
    std::vector<int4> items;
    std::vector<int> off;
    int ks[svb::kTcMaxLayers], hr[svb::kTcMaxLayers], ac[svb::kTcMaxLayers];
    for (int l = 0; l < n_layers; ++l) ks[l] = KS[l], hr[l] = has_res[l], ac[l] = accumulate[l];
    const std::vector<int> rows(rows_per_clip, rows_per_clip + B);
    SVB_TRY(svb::tc_schedule(n_layers, ks, hr, ac, Cin, B, Tq, MT, col_blocks, chain_ordered != 0, grid, &items, &off, balance_out, rows.data()));
    SVB_CHECK((int64_t)items.size() <= items_capacity, SVB_ERR_INVALID, "tc_schedule_probe_ragged: %zu items, capacity %lld", items.size(),
              (long long)items_capacity);
    for (size_t i = 0; i < items.size(); ++i) {
        int32_t *o = items_out + 5 * i;                             // layer, column block, clip, first row, tiles
        o[0] = items[i].x & 0xff, o[1] = (items[i].x >> 8) & 0xffff, o[2] = items[i].y, o[3] = items[i].z, o[4] = items[i].x >> 24;
    }
    for (int c = 0; c <= grid; ++c) off_out[c] = off[c];
    return (int64_t)items.size();
}
