// Shared definitions of the generator handle (generator.cu: forward; generator_bwd.cu: training backward).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "conv_ffma.cuh"
#include "conv_tc.cuh"
#include "nsf_source.cuh"

namespace svb {

struct HostTensor {
    std::vector<int64_t> shape;
    std::vector<float> data;
};

struct ConvLayer {          // one GEMM-shaped layer on the C4T layout
    float *w = nullptr;     // FFMA packing [KS][Cin][CoutP]
    float *b = nullptr;     // [Cout]
    TcWeights tc;           // tensor-core packing (optional)
    int Cin = 0, Cout = 0, CoutP = 0, KS = 1, dil = 1, ups_u = 0;
    double macs_per_row = 0;   // algorithmic MACs per GEMM row (true taps only)
};

struct NoiseConv {
    float *w = nullptr, *b = nullptr;
    int C = 0, K = 1, stride = 1, pad = 0;
};

struct Stage {
    int C = 0;              // channels after the upsampler
    int u = 1;
    ConvLayer up;
    NoiseConv noise;
    // resblocks[j].c1[m], c2[m]  (ResBlock2: only c1 used)
    std::vector<std::vector<ConvLayer>> c1, c2;
};

struct Tap {
    const float *p = nullptr;
    int C = 0, T = 0, Tp = 0;
    bool plain = false;     // [B][T] instead of C4T
};

// byte offsets into the workspace of one forward (in training mode this is also the tape of the backward)
struct Buffers {
    size_t mel = 0, pre = 0, har = 0, nsf = 0, sines = 0, wav = 0;
    std::vector<size_t> X, S;
    std::vector<std::vector<std::vector<size_t>>> A, R;      // [stage][ResBlock chain][dilation]
};

// dgrad twins of the ResBlock convs of one stage (flipped taps, transposed channels) + upsampler weights
// in the [K][Cout][Cin] order the strided data-gradient kernel reads
struct BwdStage {
    std::vector<std::vector<ConvLayer>> d1, d2;
    float *up_wt = nullptr;
};

// one device-side re-packing step: dst[i] = idx[i] ? nat[src][idx[i] - 1] : 0, then (optionally) the tcgen05 tiles
struct PackJob {
    std::string src;            // name of the folded tensor in the reference's layout
    float *dst = nullptr;
    int *idx = nullptr;         // nullptr: plain copy
    size_t n = 0;
    const TcWeights *tc = nullptr;
};

struct GradBuf {
    float *p = nullptr;
    size_t n = 0;
};
}  // namespace svb

struct svb_gen {
    svb_gen_config cfg{};
    int device = 0;
    bool finalized = false;
    std::map<std::string, svb::HostTensor> host_w;
    std::vector<void *> dev_allocs;

    svb::ConvLayer conv_pre;
    std::vector<svb::Stage> stages;
    float *post_wq = nullptr;
    int post_K = 7, post_C = 0;
    float *lin_w = nullptr;
    float *lin_b_dev = nullptr;     // m_source.l_linear.bias [1]
    int hop = 1;

    // workspace
    char *ws = nullptr;
    size_t ws_cap = 0;
    int ws_B = 0, ws_T = 0;
    std::map<std::string, svb::Tap> taps;
    int last_B = 0, last_T = 0;
    bool last_nsf = false;
    svb::Buffers bf;            // layout of the last forward

    // training (generator_bwd.cu): tape kept by forward, dgrad packings, gradient buffers
    bool training = false, ws_training = false, dirty = false;
    bool bwd_built = false;         // data-gradient packings + gather jobs exist (they survive set_training(0))
    std::vector<svb::BwdStage> bwd;
    float *zero_bias = nullptr;     // [max channels] zeros: the dgrad convs have no bias
    float *post_w_nat = nullptr;    // conv_post weight [C][K]
    float *post_b_dev = nullptr;
    float *grad_flat = nullptr;
    size_t grad_floats = 0;
    std::map<std::string, svb::GradBuf> grads;
    char *bws = nullptr;            // backward workspace (activation gradients)
    size_t bws_cap = 0;
    int bws_B = 0, bws_T = 0;
    int64_t bwd_launches = 0;
    std::map<std::string, svb::GradBuf> nat_dev;    // device copies of the folded tensors (svb_gen_set_weight_dev)
    std::vector<svb::PackJob> jobs;
    std::vector<void *> job_allocs;
    bool dev_dirty = false;

    // host staging (spec2wav_host)
    float *pin_in = nullptr, *pin_out = nullptr, *dev_in = nullptr, *dev_out = nullptr;
    size_t pin_in_cap = 0, pin_out_cap = 0;
    int16_t *dev_i16 = nullptr;      // int16 samples + per-clip peak (svb_gen_spec2wav_host_i16)
    size_t i16_cap = 0;

    int64_t last_launches = 0;
    double last_flops = 0;
    bool timing = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;

    // per-launch profile of the last forward (svb_gen_enable_timing(g, 2)): CUDA events around every launch
    struct LaunchRec {
        const char *name;
        cudaEvent_t e0, e1;
        double bytes, flops;
    };
    // independent ResBlock chains of a stage run side by side (SM subsets) on these streams
    cudaStream_t side[3] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_chain[3] = {nullptr, nullptr, nullptr};
    int chains = 1;     // measured on B200: side-by-side chains on SM subsets are SLOWER (7.0 vs 5.7 ms/step); kept for experiments
    double chain_bias = 4.0;

    // merged launches: the ResBlock chains of a stage step together in one persistent launch (conv_tc.cuh: TcWorkList).
    // Lists depend on the stage, the batch / length and the plan's MT; cached per (stage, chain_ordered, MT).
    bool merge = true;              // SVB_MERGE=0: one launch per convolution (round-1 schedule)
    std::map<int, svb::TcWorkList> worklists;
    std::vector<int> wl_len;        // per-clip lengths the cached lists were built for (empty: uniform batch)

    // ragged batches (svb_gen_forward_ragged): every row >= len[b] * (upsampling so far) of every activation buffer must
    // read as zero.  hw[b] = frames clip b had in the last forward since the workspace was cleared; a clip that shrinks
    // gets rows [len, hw) zeroed before the forward.
    std::vector<int> hw;
    int *rg_dev = nullptr;          // device table [len B | hw B | off B + 1] of the current ragged forward
    size_t rg_cap = 0;
    std::vector<int> cur_len;       // host copy of len (empty: uniform)
    const int *cur_len_dev = nullptr;
    double cur_frames = 0;          // sum of the clips' frames (B * T when uniform): FLOP / byte counts use valid rows only
    int cur_T = 1;

    bool profile = false;
    std::vector<LaunchRec> recs;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
};


namespace svb {
int gen_upload(svb_gen *g, const std::vector<float> &h, float **out);
int gen_get_w(svb_gen *g, const std::string &name, std::vector<int64_t> want, const HostTensor **out);
int gen_build_layers(svb_gen *g);
int gen_build_bwd_layers(svb_gen *g);      // generator_bwd.cu
}  // namespace svb
