// HiFi-GAN(-NSF) generator handle: weight packing, workspace planning and the forward schedule.
// Reference: HifiGanGenerator (modules/hifigan/hifigan.py:104-178) as driven by
// vocoders/hifigan.py:17-33 (load_model) and :55-69 (spec2wav).
#include <algorithm>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "generator.cuh"

using namespace svb;

int svb::gen_upload(svb_gen *g, const std::vector<float> &h, float **out) {
    float *d = nullptr;
    SVB_CUDA(cudaMalloc((void **)&d, std::max<size_t>(h.size(), 4) * sizeof(float)));
    SVB_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    g->dev_allocs.push_back(d);
    *out = d;
    return SVB_OK;
}

int svb::gen_get_w(svb_gen *g, const std::string &name, std::vector<int64_t> want, const HostTensor **out) {
    auto it = g->host_w.find(name);
    SVB_CHECK(it != g->host_w.end(), SVB_ERR_MISSING, "weight '%s' was never set", name.c_str());
    if (!want.empty()) {
        bool ok = it->second.shape.size() == want.size();
        for (size_t i = 0; ok && i < want.size(); ++i) ok = it->second.shape[i] == want[i];
        if (!ok) {
            std::string s;
            for (auto v : it->second.shape) s += std::to_string(v) + ",";
            std::string w;
            for (auto v : want) w += std::to_string(v) + ",";
            set_error("weight '%s' has shape [%s] but the config needs [%s]", name.c_str(), s.c_str(), w.c_str());
            return SVB_ERR_INVALID;
        }
    }
    *out = &it->second;
    return SVB_OK;
}

namespace {

int pack_conv(svb_gen *g, const std::string &prefix, int Cin, int Cout, int K, int dil, ConvLayer *L) {
    const HostTensor *w, *b;
    SVB_TRY(gen_get_w(g, prefix + ".weight", {Cout, Cin, K}, &w));
    SVB_TRY(gen_get_w(g, prefix + ".bias", {Cout}, &b));
    const std::vector<float> p = pack_conv_weights(w->data.data(), Cout, Cin, K);
    L->Cin = Cin, L->Cout = Cout, L->CoutP = Cout, L->KS = K, L->dil = dil, L->ups_u = 0;
    L->macs_per_row = (double)Cin * Cout * K;
    SVB_TRY(gen_upload(g, p, &L->w));
    SVB_TRY(gen_upload(g, b->data, &L->b));
    SVB_TRY(tc_pack_weights(p.data(), K, Cin, Cout, &L->tc, &g->dev_allocs));
    return SVB_OK;
}

int pack_convT(svb_gen *g, const std::string &prefix, int Cin, int Cout, int K, int u, int pad, ConvLayer *L) {
    const HostTensor *w, *b;
    SVB_TRY(gen_get_w(g, prefix + ".weight", {Cin, Cout, K}, &w));
    SVB_TRY(gen_get_w(g, prefix + ".bias", {Cout}, &b));
    int KS = 0;
    const std::vector<float> p = pack_convT_weights(w->data.data(), Cin, Cout, K, u, pad, &KS);
    SVB_CHECK(KS <= 11, SVB_ERR_INVALID, "upsampler %s: kernel %d / stride %d needs %d taps", prefix.c_str(), K, u, KS);
    L->Cin = Cin, L->Cout = Cout, L->CoutP = u * Cout, L->KS = KS, L->dil = 1, L->ups_u = u;
    L->macs_per_row = (double)Cin * Cout * K;    // per input row: u outputs x K/u taps
    SVB_TRY(gen_upload(g, p, &L->w));
    SVB_TRY(gen_upload(g, b->data, &L->b));
    SVB_TRY(tc_pack_weights(p.data(), KS, Cin, u * Cout, &L->tc, &g->dev_allocs));
    return SVB_OK;
}

struct Plan {
    size_t total = 0;
    size_t take(size_t bytes) {
        const size_t off = total;
        total += (bytes + 255) / 256 * 256;
        return off;
    }
};

Buffers plan_workspace(const svb_gen *g, int B, int T, size_t *total) {
    Plan p;
    Buffers b;
    b.mel = p.take(c4t_floats(B, g->cfg.n_mel, T) * 4);
    b.pre = p.take(c4t_floats(B, g->cfg.upsample_initial_channel, T) * 4);
    b.har = p.take((size_t)B * T * g->hop * 4);
    b.nsf = p.take(nsf_workspace_bytes(B, T, g->hop));
    int Ti = T;
    for (auto &s : g->stages) {
        Ti *= s.u;
        const size_t n = c4t_floats(B, s.C, Ti) * 4;
        b.X.push_back(p.take(n)), b.S.push_back(p.take(n));
        b.A.emplace_back(), b.R.emplace_back();
        for (int j = 0; j < g->cfg.n_resblock_kernels; ++j) {
            // inference: one A / R buffer per chain, reused by every dilation; training: every conv input is kept (the tape)
            std::vector<size_t> a(g->cfg.n_dilations), r(g->cfg.n_dilations);
            for (int m = 0; m < g->cfg.n_dilations; ++m) {
                a[m] = (m == 0 || g->training) ? p.take(n) : a[0];
                r[m] = (m == 0 || g->training) ? p.take(n) : r[0];
            }
            b.A.back().push_back(a), b.R.back().push_back(r);
        }
    }
    if (g->training) {
        b.sines = p.take((size_t)B * T * g->hop * 9 * 4);
        b.wav = p.take((size_t)B * T * g->hop * 4);
    }
    *total = p.total;
    return b;
}

cudaEvent_t prof_event(svb_gen *g) {
    if (g->ev_used == g->ev_pool.size()) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        g->ev_pool.push_back(e);
    }
    return g->ev_pool[g->ev_used++];
}
// wraps one launch with events when profiling; `bytes` = algorithmic HBM bytes of the launch
struct ProfScope {
    svb_gen *g;
    cudaStream_t st;
    cudaEvent_t e1 = nullptr;
    ProfScope(svb_gen *g_, cudaStream_t st_, const char *name, double bytes, double flops) : g(g_), st(st_) {
        if (!g->profile) return;
        cudaEvent_t e0 = prof_event(g);
        e1 = prof_event(g);
        cudaEventRecord(e0, st);
        g->recs.push_back({name, e0, e1, bytes, flops});
    }
    ~ProfScope() {
        if (e1) cudaEventRecord(e1, st);
    }
};

// valid GEMM rows of a layer with Tq rows per clip at the longest clip (= B * Tq for a uniform batch)
double valid_rows_total(const svb_gen *g, int Tq) { return g->cur_frames * (double)(Tq / g->cur_T); }
// host [B] valid rows per clip at Tq rows for the longest clip; empty for a uniform batch
std::vector<int> clip_rows(const svb_gen *g, int Tq) {
    std::vector<int> r(g->cur_len);
    for (int &v : r) v *= Tq / g->cur_T;
    return r;
}

int run_conv(svb_gen *g, const ConvLayer &L, const float *in, int in_Tp, float *out, int out_Tp, const float *res,
             int B, int Tq, float in_slope, float scale, int accumulate, cudaStream_t st, int max_ctas = 0) {
    const double rows = valid_rows_total(g, Tq);
    g->last_launches += 1;
    g->last_flops += 2.0 * L.macs_per_row * rows;
    const bool tc = g->cfg.precision != SVB_PREC_FP32 && L.tc.ok;
    const double rows_out = rows * (L.ups_u > 0 ? L.ups_u : 1);
    // layer-streaming bytes (SURVEY 8(d)): input once, output once, residual / accumulated sum once more each
    const double bytes = 4.0 * (rows * L.Cin + rows_out * L.Cout * (1 + (res ? 1 : 0) + (accumulate ? 1 : 0)));
    ProfScope ps(g, st, tc ? (L.ups_u ? "conv1d_c4_tc (upsampler)" : "conv1d_c4_tc (resblock)") : "conv1d_c4_ffma", bytes,
                 2.0 * L.macs_per_row * rows);
    ConvArgs a;
    a.in = in, a.w = L.w, a.bias = L.b, a.res = res, a.out = out;
    a.B = B, a.Cin = L.Cin, a.in_Tp = in_Tp, a.Cout = L.Cout, a.out_Tp = out_Tp, a.CoutP = L.CoutP, a.Tq = Tq;
    a.KS = L.KS, a.dil = L.dil, a.ups_u = L.ups_u, a.in_slope = in_slope, a.out_scale = scale, a.accumulate = accumulate;
    a.rows = g->cur_len_dev, a.rows_mul = Tq / g->cur_T;
    if (g->cfg.precision != SVB_PREC_FP32 && tc_supported(L.tc, a)) return launch_conv_tc(L.tc, a, g->cfg.precision, st, max_ctas);
    return launch_conv_ffma(a, st);
}

// One merged launch over the nk layers `Ls` (same shape class): layer j reads in[j], writes out[j], adds res[j].
// chain_ordered: later layers accumulate into the output of earlier ones (the ResBlock sum), see TcWorkList.
int run_conv_multi(svb_gen *g, int stage, int nk, const ConvLayer *const *Ls, const float *const *in, float *const *out,
                   const float *const *res, const float *scale, const int *accumulate, bool chain_ordered, int B, int Tq, int Tp,
                   float in_slope, cudaStream_t st) {
    ConvArgs a[kTcMaxLayers];
    const TcWeights *w[kTcMaxLayers];
    double bytes = 0, flops = 0;
    const double rows = valid_rows_total(g, Tq);
    for (int j = 0; j < nk; ++j) {
        const ConvLayer &L = *Ls[j];
        a[j].in = in[j], a[j].w = L.w, a[j].bias = L.b, a[j].res = res[j], a[j].out = out[j];
        a[j].B = B, a[j].Cin = L.Cin, a[j].in_Tp = Tp, a[j].Cout = L.Cout, a[j].out_Tp = Tp, a[j].CoutP = L.CoutP, a[j].Tq = Tq;
        a[j].KS = L.KS, a[j].dil = L.dil, a[j].ups_u = 0, a[j].in_slope = in_slope, a[j].out_scale = scale[j], a[j].accumulate = accumulate[j];
        a[j].rows = g->cur_len_dev, a[j].rows_mul = Tq / g->cur_T;
        w[j] = &L.tc;
        bytes += 4.0 * (rows * L.Cin + rows * L.Cout * (1 + (res[j] ? 1 : 0) + (accumulate[j] ? 1 : 0)));
        flops += 2.0 * L.macs_per_row * rows;
    }
    g->last_launches += 1;
    g->last_flops += flops;
    ProfScope ps(g, st, "conv1d_c4_tc (resblock)", bytes, flops);
    // the list depends on the plan (MT) of this layer set: try the cached one, rebuild on a plan mismatch
    for (int attempt = 0; attempt < 2; ++attempt) {
        const int key = stage * 4 + (chain_ordered ? 2 : 0) + attempt;
        TcWorkList &wl = g->worklists[key];
        if (!wl.valid) {
            const std::vector<int> rh = clip_rows(g, Tq);
            SVB_TRY(tc_worklist_build(nk, w, a, g->cfg.precision, chain_ordered, &wl, rh.empty() ? nullptr : rh.data(), st));
        }
        const int rc = launch_conv_tc_multi(nk, w, a, g->cfg.precision, st, wl);
        if (rc != SVB_ERR_STATE) return rc;
    }
    set_error("merged launch: no cached work list matches the plan of stage %d", stage);
    return SVB_ERR_STATE;
}

// The one generator forward.  lens == nullptr: B clips of T frames.  lens = host [B] (1 <= lens[b] <= T): a ragged batch in the
// padded layout (clip b's frames 0 .. lens[b] - 1; nothing past them is read, wav past lens[b] * hop is written as 0), or, with
// `packed`, clip after clip in mel [sum lens, n_mel] (frame-major) / f0 [sum lens] / wav [sum lens * hop].
int forward_impl(svb_gen *g, const float *mel, bool mel_frame_major, const float *f0, const float *rand_ini,
                 const float *noise, uint64_t seed, int B, int T, float *wav, cudaStream_t st, const int32_t *lens = nullptr,
                 bool packed = false) {
    SVB_CHECK(g && g->finalized, SVB_ERR_STATE, "generator: forward before finalize");
    SVB_CHECK(!g->dirty, SVB_ERR_STATE, "generator: weights were set after finalize; call svb_gen_update_weights first");
    SVB_CHECK(mel && wav && B > 0 && T > 0, SVB_ERR_INVALID, "generator: null buffer or empty batch (B %d T %d)", B, T);
    SVB_CHECK(!f0 || g->cfg.use_pitch_embed, SVB_ERR_INVALID, "generator: f0 given but use_pitch_embed is off");
    SVB_CHECK((rand_ini == nullptr) == (noise == nullptr), SVB_ERR_INVALID,
              "generator: rand_ini and noise must be given together");
    SVB_CHECK(!lens || !g->training, SVB_ERR_INVALID,
              "generator: a ragged batch is inference only (training takes clips of equal length)");
    SVB_CHECK(!packed || (lens && mel_frame_major && !noise), SVB_ERR_INVALID, "generator: bad packed-layout call");
    SVB_CUDA(cudaSetDevice(g->device));
    size_t need = 0;
    Buffers bf = plan_workspace(g, B, T, &need);
    if (need > g->ws_cap) {
        if (g->ws) SVB_CUDA(cudaFree(g->ws));
        g->ws = nullptr, g->ws_cap = 0;
        SVB_CUDA(cudaMalloc((void **)&g->ws, need));
        g->ws_cap = need, g->ws_B = 0;
    }
    std::vector<int> len;
    if (lens) len.assign(lens, lens + B);
    if (g->ws_B != B || g->ws_T != T || len != g->wl_len) {            // the work lists depend on the batch and its lengths
        for (auto &kv : g->worklists) kv.second.valid = false;
        g->wl_len = len;
    }
    if (g->ws_B != B || g->ws_T != T || g->ws_training != g->training) {   // new layout: rebuild the zero padding of every buffer
        SVB_CUDA(cudaMemsetAsync(g->ws, 0, need, st));
        g->ws_B = B, g->ws_T = T, g->ws_training = g->training;
        g->hw.assign(B, 0);
    }
    g->cur_len = len, g->cur_len_dev = nullptr, g->cur_T = T, g->cur_frames = (double)B * T;
    Ragged rg;
    int stale_rows = 0;                         // longest stale tail (frames) a shrunk clip left behind
    if (lens) {
        // device table [len B | hw B | off B + 1], grow-only; uploaded from pageable memory (staged before the call returns)
        std::vector<int> tab(3 * (size_t)B + 1);
        double frames = 0;
        for (int b = 0; b < B; ++b) {
            tab[b] = len[b], tab[B + b] = g->hw[b], tab[2 * B + b] = (int)frames;
            stale_rows = std::max(stale_rows, g->hw[b] - len[b]);
            frames += len[b];
        }
        tab[3 * B] = (int)frames;
        if (tab.size() > g->rg_cap) {
            if (g->rg_dev) SVB_CUDA(cudaFree(g->rg_dev));
            g->rg_dev = nullptr, g->rg_cap = 0;
            SVB_CUDA(cudaMalloc((void **)&g->rg_dev, tab.size() * sizeof(int)));
            g->rg_cap = tab.size();
        }
        SVB_CUDA(cudaMemcpyAsync(g->rg_dev, tab.data(), tab.size() * sizeof(int), cudaMemcpyHostToDevice, st));
        g->cur_len_dev = g->rg_dev, g->cur_frames = frames;
        rg.len = g->rg_dev, rg.off = packed ? g->rg_dev + 2 * B : nullptr;
    }
    for (int b = 0; b < B; ++b) g->hw[b] = lens ? len[b] : T;
    g->bf = bf, g->last_T = T, g->last_nsf = f0 != nullptr;
    g->last_launches = 0, g->last_flops = 0, g->last_B = B;
    g->taps.clear();
    g->recs.clear(), g->ev_used = 0;
    if (g->timing) SVB_CUDA(cudaEventRecord(g->ev0, st));

    auto F = [&](size_t off) { return reinterpret_cast<float *>(g->ws + off); };
    const int n_mel = g->cfg.n_mel, C0 = g->cfg.upsample_initial_channel;
    const int Tp0 = c4t_rows(T);
    const double frames = g->cur_frames;
    if (stale_rows > 0) {
        // a clip shrank since the last forward: its rows [len, hw) of every buffer a conv reads past the clip's end
        // go back to zero (the mel buffer is rewritten in full below)
        std::vector<ZeroSeg> segs;
        segs.push_back({F(bf.pre), c4t_groups(C0), Tp0, 1});
        int mul = 1, max_rows = stale_rows;
        for (size_t i = 0; i < g->stages.size(); ++i) {
            const Stage &s = g->stages[i];
            mul *= s.u;
            const int Tip = c4t_rows(T * mul), gr = c4t_groups(s.C);
            std::vector<size_t> offs = {bf.X[i], bf.S[i]};
            for (auto &v : bf.A[i]) offs.insert(offs.end(), v.begin(), v.end());
            for (auto &v : bf.R[i]) offs.insert(offs.end(), v.begin(), v.end());
            std::sort(offs.begin(), offs.end());
            offs.erase(std::unique(offs.begin(), offs.end()), offs.end());
            for (size_t o : offs) segs.push_back({F(o), gr, Tip, mul});
            max_rows = std::max(max_rows, stale_rows * mul);
        }
        ProfScope ps(g, st, "zero stale rows", 0, 0);
        for (size_t i0 = 0; i0 < segs.size(); i0 += kMaxZeroSegs)
            SVB_TRY(launch_zero_tails(segs.data() + i0, (int)std::min<size_t>(kMaxZeroSegs, segs.size() - i0), B, g->rg_dev,
                                      g->rg_dev + B, max_rows, st));
        g->last_launches += (int64_t)((segs.size() + kMaxZeroSegs - 1) / kMaxZeroSegs);
    }
    {
        ProfScope ps(g, st, "mel layout", 8.0 * n_mel * frames, 0);
        if (mel_frame_major) SVB_TRY(launch_btc_to_c4t(mel, F(bf.mel), B, n_mel, T, Tp0, st, rg));
        else SVB_TRY(launch_nct_to_c4t(mel, F(bf.mel), B, n_mel, T, Tp0, st, rg));
    }
    g->last_launches += 1;

    const int Tw = T * g->hop;
    float *har = nullptr;
    bool har_on_side = false;
    if (f0) {
        // The NSF source only meets the main chain at the first noise_conv_add: run it on a side stream
        // so it overlaps conv_pre and the first upsampler.
        har = F(bf.har);
        har_on_side = !g->profile;
        cudaStream_t ns = har_on_side ? g->side[0] : st;
        if (har_on_side) {
            SVB_CUDA(cudaEventRecord(g->ev_fork, st));
            SVB_CUDA(cudaStreamWaitEvent(ns, g->ev_fork, 0));
        }
        int l = 0;
        {
            const double samples = frames * g->hop;
            ProfScope ps(g, ns, "nsf source (4 kernels)", 4.0 * (frames + samples * (noise ? 10 : 1)), 60.0 * samples * 9);
            SVB_TRY(launch_nsf_source(f0, rand_ini, noise, seed, B, T, g->hop, (float)g->cfg.audio_sample_rate, g->lin_w,
                                      g->lin_b_dev, g->ws + bf.nsf, har, g->training ? F(bf.sines) : nullptr, ns, &l, rg.len, rg.off));
        }
        if (har_on_side) SVB_CUDA(cudaEventRecord(g->ev_chain[0], ns));
        g->last_launches += l;
        g->taps["har_source"] = Tap{har, 1, Tw, 0, true};
    }

    SVB_TRY(run_conv(g, g->conv_pre, F(bf.mel), Tp0, F(bf.pre), Tp0, nullptr, B, T, 1.f, 1.f, 0, st));
    g->taps["conv_pre"] = Tap{F(bf.pre), C0, T, Tp0, false};

    const float *x_in = F(bf.pre);
    int Tin = T, Tin_p = Tp0;
    const int nk = g->cfg.n_resblock_kernels, nd = g->cfg.n_dilations;
    for (size_t i = 0; i < g->stages.size(); ++i) {
        Stage &s = g->stages[i];
        const int Ti = Tin * s.u, Tip = c4t_rows(Ti);
        float *X = F(bf.X[i]), *S = F(bf.S[i]);
        // x = ups[i](leaky_relu(x, 0.1))            hifigan.py:153-154
        SVB_TRY(run_conv(g, s.up, x_in, Tin_p, X, Tip, nullptr, B, Tin, 0.1f, 1.f, 0, st));
        if (f0) {                                   // x = x + noise_convs[i](har_source)   :155-157
            if (har_on_side && i == 0) SVB_CUDA(cudaStreamWaitEvent(st, g->ev_chain[0], 0));
            const double rows = valid_rows_total(g, Ti);
            ProfScope ps(g, st, "noise_conv_add", 4.0 * (2.0 * rows * s.C + frames * g->hop), 2.0 * rows * s.C * s.noise.K);
            SVB_TRY(launch_noise_conv_add(X, B, s.C, Ti, Tip, har, Tw, s.noise.w, s.noise.b, s.noise.K, s.noise.stride,
                                          s.noise.pad, st, rg, Ti / T, g->hop));
            g->last_launches += 1;
            g->last_flops += 2.0 * rows * s.C * s.noise.K;
        }
        g->taps["ups" + std::to_string(i)] = Tap{X, s.C, Ti, Tip, false};
        // xs = sum_j resblocks[i*nk + j](x) ; x = xs / nk      :158-164
        // The nk ResBlocks only share their input: each chain runs on its own stream and SM subset, which
        // amortises the per-launch fill/drain of the persistent kernels; the final convs (which add
        // into S) are ordered by events.
        const bool par = g->chains > 1 && nk > 1 && nk <= 3 && g->cfg.precision != SVB_PREC_FP32 && !g->profile;
        const int sms = 148;
        // merged schedule: step m of all nk chains in ONE persistent launch (the chains only share their input)
        bool merged = g->merge && !par && nk > 1 && nk <= kTcMaxLayers && g->cfg.precision != SVB_PREC_FP32 &&
                      s.c1[0][0].tc.ok;
        if (merged) {
            const std::vector<int> rh = clip_rows(g, Ti);
            merged = tc_merge_fits(nk, B, Ti, s.C, s.c1[0][0].tc.n_tile, rh.empty() ? nullptr : rh.data());
        }
        for (int j = 0; merged && j < nk; ++j)
            for (int m = 0; m < nd; ++m) {
                ConvArgs probe;
                probe.Cin = s.C, probe.Cout = s.C, probe.CoutP = s.C, probe.KS = s.c1[j][m].KS, probe.dil = s.c1[j][m].dil, probe.ups_u = 0;
                probe.bias = s.c1[j][m].b, probe.cin_blk = 0;
                merged = merged && tc_supported(s.c1[j][m].tc, probe) && s.c1[j][m].tc.n_tile == s.c1[0][0].tc.n_tile;
                if (g->cfg.resblock == 1) merged = merged && s.c2[j][m].tc.ok && s.c2[j][m].tc.n_tile == s.c1[0][0].tc.n_tile;
            }
        if (merged) {
            for (int m = 0; m < nd; ++m) {
                const bool last = m == nd - 1;
                const ConvLayer *L1[kTcMaxLayers], *L2[kTcMaxLayers];
                const float *xin[kTcMaxLayers], *ain[kTcMaxLayers], *none[kTcMaxLayers];
                float *aout[kTcMaxLayers], *dst[kTcMaxLayers];
                float one[kTcMaxLayers], scl[kTcMaxLayers];
                int zero[kTcMaxLayers], acc[kTcMaxLayers];
                for (int j = 0; j < nk; ++j) {
                    L1[j] = &s.c1[j][m], none[j] = nullptr, one[j] = 1.f, zero[j] = 0;
                    scl[j] = last ? 1.f / nk : 1.f, acc[j] = (last && j > 0) ? 1 : 0;
                    if (g->cfg.resblock == 1) {                 // ResBlock1.forward :54-61
                        L2[j] = &s.c2[j][m];
                        xin[j] = m == 0 ? X : F(bf.R[i][j][m - 1]);
                        aout[j] = F(bf.A[i][j][m]), ain[j] = aout[j];
                        dst[j] = last ? S : F(bf.R[i][j][m]);
                    } else {                                    // ResBlock2.forward :81-86 (never in place: ping-pong A / R)
                        xin[j] = m == 0 ? X : (m % 2 ? F(bf.R[i][j][m - 1]) : F(bf.A[i][j][m - 1]));
                        dst[j] = last ? S : (m % 2 ? F(bf.A[i][j][m]) : F(bf.R[i][j][m]));
                    }
                }
                if (g->cfg.resblock == 1) {
                    SVB_TRY(run_conv_multi(g, (int)i, nk, L1, xin, aout, none, one, zero, false, B, Ti, Tip, 0.1f, st));
                    SVB_TRY(run_conv_multi(g, (int)i, nk, L2, ain, dst, xin, scl, acc, last, B, Ti, Tip, 0.1f, st));
                } else {
                    SVB_TRY(run_conv_multi(g, (int)i, nk, L1, xin, dst, xin, scl, acc, last, B, Ti, Tip, 0.1f, st));
                }
            }
        }
        if (par) SVB_CUDA(cudaEventRecord(g->ev_fork, st));
        for (int j = 0; j < nk && !merged; ++j) {
            cudaStream_t cs = par ? g->side[j] : st;
            // SM share of a chain ~ its cost: kernel size plus a constant for the memory-bound part
            int cap = 0;
            if (par) {
                double wsum = 0, wj = 0;
                for (int jj = 0; jj < nk; ++jj) {
                    const double wv = g->cfg.resblock_kernel_sizes[jj] + g->chain_bias;
                    wsum += wv;
                    if (jj == j) wj = wv;
                }
                cap = std::max(8, (int)(sms * wj / wsum + 0.5));
                if (g->chains == 2) cap = 0;    // full grids on every stream: the block scheduler interleaves the chains' CTAs
            }
            if (par) SVB_CUDA(cudaStreamWaitEvent(cs, g->ev_fork, 0));
            for (int m = 0; m < nd; ++m) {
                float *A = F(bf.A[i][j][m]);
                const float *xin = m == 0 ? X : F(bf.R[i][j][m - 1]);
                const bool last = m == nd - 1;
                float *dst = last ? S : F(bf.R[i][j][m]);
                const float scale = last ? 1.f / nk : 1.f;
                const int accum = (last && j > 0) ? 1 : 0;
                if (g->cfg.resblock == 1) {         // ResBlock1.forward :54-61
                    SVB_TRY(run_conv(g, s.c1[j][m], xin, Tip, A, Tip, nullptr, B, Ti, 0.1f, 1.f, 0, cs, cap));
                    if (par && last && j > 0) SVB_CUDA(cudaStreamWaitEvent(cs, g->ev_chain[j - 1], 0));
                    SVB_TRY(run_conv(g, s.c2[j][m], A, Tip, dst, Tip, xin, B, Ti, 0.1f, scale, accum, cs, cap));
                } else {                            // ResBlock2.forward :81-86 (never in place: ping-pong A / R)
                    const float *xin2 = m == 0 ? X : (m % 2 ? F(bf.R[i][j][m - 1]) : F(bf.A[i][j][m - 1]));
                    float *dst2 = last ? S : (m % 2 ? F(bf.A[i][j][m]) : F(bf.R[i][j][m]));
                    if (par && last && j > 0) SVB_CUDA(cudaStreamWaitEvent(cs, g->ev_chain[j - 1], 0));
                    SVB_TRY(run_conv(g, s.c1[j][m], xin2, Tip, dst2, Tip, xin2, B, Ti, 0.1f, scale, accum, cs, cap));
                }
            }
            if (par) SVB_CUDA(cudaEventRecord(g->ev_chain[j], cs));
        }
        if (par) SVB_CUDA(cudaStreamWaitEvent(st, g->ev_chain[nk - 1], 0));
        g->taps["stage" + std::to_string(i)] = Tap{S, s.C, Ti, Tip, false};
        x_in = S, Tin = Ti, Tin_p = Tip;
    }
    // x = tanh(conv_post(leaky_relu(x)))   default slope 0.01   :165-167
    {
        const double rows = valid_rows_total(g, Tin);
        ProfScope ps(g, st, "conv_post_tanh", 4.0 * rows * (g->post_C + 1.0), 2.0 * rows * g->post_C * g->post_K);
        SVB_TRY(launch_conv_post_tanh(x_in, B, g->post_C, Tin, Tin_p, g->post_wq, g->post_b_dev, g->post_K, 0.01f, wav, st, rg,
                                      Tin / T));
    }
    g->last_launches += 1;
    g->last_flops += 2.0 * valid_rows_total(g, Tin) * g->post_C * g->post_K;
    if (g->training) SVB_CUDA(cudaMemcpyAsync(F(bf.wav), wav, (size_t)B * Tw * 4, cudaMemcpyDeviceToDevice, st));
    if (g->timing) SVB_CUDA(cudaEventRecord(g->ev1, st));
    return SVB_OK;
}

}  // namespace

extern "C" int svb_gen_create(const svb_gen_config *cfg, int device, svb_gen_t **out) {
    SVB_CHECK(cfg && out, SVB_ERR_INVALID, "gen_create: null argument");
    SVB_CHECK(cfg->n_ups >= 1 && cfg->n_ups <= SVB_MAX_UPS, SVB_ERR_INVALID, "gen_create: n_ups %d out of range", cfg->n_ups);
    SVB_CHECK(cfg->n_resblock_kernels >= 1 && cfg->n_resblock_kernels <= SVB_MAX_RBK, SVB_ERR_INVALID,
              "gen_create: n_resblock_kernels %d out of range", cfg->n_resblock_kernels);
    SVB_CHECK(cfg->n_dilations >= 1 && cfg->n_dilations <= SVB_MAX_DIL, SVB_ERR_INVALID, "gen_create: n_dilations %d",
              cfg->n_dilations);
    SVB_CHECK(cfg->resblock == 1 || cfg->resblock == 2, SVB_ERR_INVALID, "gen_create: resblock must be 1 or 2");
    SVB_CHECK(cfg->n_mel > 0 && cfg->n_mel % 4 == 0, SVB_ERR_INVALID, "gen_create: n_mel %d must be a multiple of 4",
              cfg->n_mel);
    SVB_CHECK(cfg->precision >= 0 && cfg->precision <= 3, SVB_ERR_INVALID, "gen_create: bad precision %d", cfg->precision);
    const int cfin = cfg->upsample_initial_channel >> cfg->n_ups;
    SVB_CHECK(cfin >= 4 && (cfin << cfg->n_ups) == cfg->upsample_initial_channel && cfin % 4 == 0, SVB_ERR_INVALID,
              "gen_create: upsample_initial_channel %d must stay a multiple of 4 after %d halvings",
              cfg->upsample_initial_channel, cfg->n_ups);
    for (int j = 0; j < cfg->n_resblock_kernels; ++j) {
        const int k = cfg->resblock_kernel_sizes[j];
        SVB_CHECK(k % 2 == 1 && k >= 1 && k <= 11, SVB_ERR_INVALID, "gen_create: resblock kernel %d unsupported", k);
        for (int m = 0; m < cfg->n_dilations; ++m)
            SVB_CHECK((k - 1) / 2 * cfg->resblock_dilation_sizes[j][m] <= kPad && cfg->resblock_dilation_sizes[j][m] >= 1,
                      SVB_ERR_INVALID, "gen_create: kernel %d dilation %d exceeds the %d-row halo", k,
                      cfg->resblock_dilation_sizes[j][m], kPad);
    }
    int count = 0;
    SVB_CUDA(cudaGetDeviceCount(&count));
    SVB_CHECK(device >= 0 && device < count, SVB_ERR_INVALID, "gen_create: device %d of %d", device, count);
    SVB_CUDA(cudaSetDevice(device));
    svb_gen *g = new (std::nothrow) svb_gen();
    SVB_CHECK(g, SVB_ERR_NOMEM, "gen_create: out of host memory");
    g->cfg = *cfg, g->device = device;
    g->hop = 1;
    for (int i = 0; i < cfg->n_ups; ++i) g->hop *= cfg->upsample_rates[i];
    SVB_CUDA(cudaEventCreate(&g->ev0));
    SVB_CUDA(cudaEventCreate(&g->ev1));
    SVB_CUDA(cudaEventCreateWithFlags(&g->ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < 3; ++i) {
        SVB_CUDA(cudaStreamCreateWithFlags(&g->side[i], cudaStreamNonBlocking));
        SVB_CUDA(cudaEventCreateWithFlags(&g->ev_chain[i], cudaEventDisableTiming));
    }
    if (const char *e = getenv("SVB_CHAINS")) g->chains = atoi(e);
    if (const char *e = getenv("SVB_MERGE")) g->merge = atoi(e) != 0;
    if (const char *e = getenv("SVB_CHAIN_BIAS")) g->chain_bias = atof(e);
    *out = g;
    return SVB_OK;
}

extern "C" void svb_gen_destroy(svb_gen_t *g) {
    if (!g) return;
    cudaSetDevice(g->device);
    for (void *p : g->dev_allocs) cudaFree(p);
    for (auto &kv : g->worklists) tc_worklist_free(&kv.second);
    if (g->ws) cudaFree(g->ws);
    if (g->rg_dev) cudaFree(g->rg_dev);
    if (g->bws) cudaFree(g->bws);
    for (void *p : g->job_allocs) cudaFree(p);
    for (auto &kv : g->nat_dev) cudaFree(kv.second.p);
    if (g->grad_flat) cudaFree(g->grad_flat);
    if (g->pin_in) cudaFreeHost(g->pin_in);
    if (g->pin_out) cudaFreeHost(g->pin_out);
    if (g->dev_in) cudaFree(g->dev_in);
    if (g->dev_out) cudaFree(g->dev_out);
    if (g->dev_i16) cudaFree(g->dev_i16);
    for (cudaEvent_t e : g->ev_pool) cudaEventDestroy(e);
    for (int i = 0; i < 3; ++i) {
        if (g->side[i]) cudaStreamDestroy(g->side[i]);
        if (g->ev_chain[i]) cudaEventDestroy(g->ev_chain[i]);
    }
    if (g->ev_fork) cudaEventDestroy(g->ev_fork);
    if (g->ev0) cudaEventDestroy(g->ev0);
    if (g->ev1) cudaEventDestroy(g->ev1);
    delete g;
}

extern "C" int svb_gen_set_weight(svb_gen_t *g, const char *name, const float *data, const int64_t *shape, int32_t ndim) {
    SVB_CHECK(g && name && data && shape && ndim >= 1 && ndim <= 4, SVB_ERR_INVALID, "set_weight: bad argument");
    SVB_CHECK(!g->finalized || g->training, SVB_ERR_STATE, "set_weight('%s') after finalize (only a training handle takes new weights)", name);
    if (g->finalized) g->dirty = true;
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; ++i) {
        SVB_CHECK(shape[i] > 0, SVB_ERR_INVALID, "set_weight('%s'): non-positive dim", name);
        t.shape.push_back(shape[i]);
        n *= (size_t)shape[i];
    }
    t.data.assign(data, data + n);
    g->host_w[name] = std::move(t);
    return SVB_OK;
}

// (re)build every device packing from the host copies of the weights
int svb::gen_build_layers(svb_gen *g) {
    SVB_CUDA(cudaSetDevice(g->device));
    for (void *p : g->dev_allocs) cudaFree(p);
    g->dev_allocs.clear();
    g->stages.clear();
    g->conv_pre = ConvLayer();
    const svb_gen_config &c = g->cfg;
    const int C0 = c.upsample_initial_channel;
    SVB_TRY(pack_conv(g, "conv_pre", c.n_mel, C0, 7, 1, &g->conv_pre));          // hifigan.py:118
    int cin = C0;
    g->stages.resize(c.n_ups);
    for (int i = 0; i < c.n_ups; ++i) {
        Stage &s = g->stages[i];
        const int u = c.upsample_rates[i], k = c.upsample_kernel_sizes[i];
        s.C = cin / 2, s.u = u;
        SVB_CHECK(k >= u && (k - u) % 2 == 0, SVB_ERR_INVALID, "upsampler %d: kernel %d / rate %d unsupported", i, k, u);
        SVB_TRY(pack_convT(g, "ups." + std::to_string(i), cin, s.C, k, u, (k - u) / 2, &s.up));   // :122-125
        if (c.use_pitch_embed) {                                                                   // :126-132
            int stride = 1;
            for (int r = i + 1; r < c.n_ups; ++r) stride *= c.upsample_rates[r];
            const bool last = i + 1 == c.n_ups;
            s.noise.C = s.C, s.noise.K = last ? 1 : 2 * stride, s.noise.stride = last ? 1 : stride;
            s.noise.pad = last ? 0 : stride / 2;
            const HostTensor *w, *b;
            SVB_TRY(gen_get_w(g, "noise_convs." + std::to_string(i) + ".weight", {s.C, 1, s.noise.K}, &w));
            SVB_TRY(gen_get_w(g, "noise_convs." + std::to_string(i) + ".bias", {s.C}, &b));
            std::vector<float> wt((size_t)s.noise.K * s.C);                       // [C][1][K] -> [K][C]
            for (int ch = 0; ch < s.C; ++ch)
                for (int j = 0; j < s.noise.K; ++j) wt[(size_t)j * s.C + ch] = w->data[(size_t)ch * s.noise.K + j];
            SVB_TRY(gen_upload(g, wt, &s.noise.w));
            SVB_TRY(gen_upload(g, b->data, &s.noise.b));
        }
        s.c1.resize(c.n_resblock_kernels), s.c2.resize(c.n_resblock_kernels);
        for (int j = 0; j < c.n_resblock_kernels; ++j) {
            const int n = i * c.n_resblock_kernels + j, rk = c.resblock_kernel_sizes[j];
            s.c1[j].resize(c.n_dilations), s.c2[j].resize(c.n_dilations);
            for (int m = 0; m < c.n_dilations; ++m) {
                const int d = c.resblock_dilation_sizes[j][m];
                const std::string base = "resblocks." + std::to_string(n);
                if (c.resblock == 1) {
                    SVB_TRY(pack_conv(g, base + ".convs1." + std::to_string(m), s.C, s.C, rk, d, &s.c1[j][m]));
                    SVB_TRY(pack_conv(g, base + ".convs2." + std::to_string(m), s.C, s.C, rk, 1, &s.c2[j][m]));
                } else {
                    SVB_TRY(pack_conv(g, base + ".convs." + std::to_string(m), s.C, s.C, rk, d, &s.c1[j][m]));
                }
            }
        }
        cin = s.C;
    }
    {   // conv_post: Conv1d(ch, 1, 7, padding 3)   :140
        const HostTensor *w, *b;
        SVB_TRY(gen_get_w(g, "conv_post.weight", {1, cin, 7}, &w));
        SVB_TRY(gen_get_w(g, "conv_post.bias", {1}, &b));
        std::vector<float> p((size_t)cin * 7);
        for (int cq = 0; cq < cin / 4; ++cq)
            for (int k = 0; k < 7; ++k)
                for (int e = 0; e < 4; ++e) p[((size_t)cq * 7 + k) * 4 + e] = w->data[(size_t)(cq * 4 + e) * 7 + k];
        SVB_TRY(gen_upload(g, p, &g->post_wq));
        SVB_TRY(gen_upload(g, b->data, &g->post_b_dev));
        g->post_K = 7, g->post_C = cin;
    }
    if (c.use_pitch_embed) {   // m_source.l_linear: Linear(9, 1)   source.py:378
        const HostTensor *w, *b;
        SVB_TRY(gen_get_w(g, "m_source.l_linear.weight", {1, 9}, &w));
        SVB_TRY(gen_get_w(g, "m_source.l_linear.bias", {1}, &b));
        SVB_TRY(gen_upload(g, w->data, &g->lin_w));
        SVB_TRY(gen_upload(g, b->data, &g->lin_b_dev));
    }
    return SVB_OK;
}

extern "C" int svb_gen_finalize(svb_gen_t *g) {
    SVB_CHECK(g, SVB_ERR_INVALID, "finalize: null handle");
    SVB_CHECK(!g->finalized, SVB_ERR_STATE, "finalize called twice");
    SVB_TRY(gen_build_layers(g));
    g->finalized = true;        // host copies are kept: training re-packs from them after every optimizer step
    return SVB_OK;
}

extern "C" int svb_gen_set_precision(svb_gen_t *g, int32_t precision) {
    SVB_CHECK(g && precision >= 0 && precision <= 3, SVB_ERR_INVALID, "set_precision: bad argument");
    g->cfg.precision = precision;
    return SVB_OK;
}

extern "C" int svb_gen_forward(svb_gen_t *g, const float *mel_dev, const float *f0_dev, const float *rand_ini_dev,
                               const float *noise_dev, uint64_t seed, int32_t B, int32_t T, float *wav_dev, void *stream) {
    return forward_impl(g, mel_dev, false, f0_dev, rand_ini_dev, noise_dev, seed, B, T, wav_dev, as_stream(stream));
}

namespace {
// lengths of a ragged batch: every clip 1 .. T_max frames (T_max <= 0: no upper bound); checked before any CUDA call
int check_lengths(const char *what, const int32_t *lens, int B, int T_max) {
    SVB_CHECK(lens, SVB_ERR_INVALID, "%s: lengths is NULL", what);
    SVB_CHECK(B > 0, SVB_ERR_INVALID, "%s: empty batch (B %d)", what, B);
    long long frames = 0;
    for (int b = 0; b < B; ++b) {
        SVB_CHECK(lens[b] >= 1 && (T_max <= 0 || lens[b] <= T_max), SVB_ERR_INVALID,
                  "%s: length %d of clip %d is outside [1, T_max %d]", what, lens[b], b, T_max);
        frames += lens[b];
    }
    SVB_CHECK(frames < (1ll << 31) / 4096, SVB_ERR_INVALID, "%s: %lld frames in one batch", what, frames);
    return SVB_OK;
}
}  // namespace

extern "C" int svb_gen_forward_ragged(svb_gen_t *g, const float *mel_dev, const float *f0_dev, const int32_t *lengths_host,
                                      const float *rand_ini_dev, const float *noise_dev, uint64_t seed, int32_t B, int32_t T_max,
                                      float *wav_dev, void *stream) {
    SVB_CHECK(T_max > 0, SVB_ERR_INVALID, "gen_forward_ragged: T_max %d", T_max);
    SVB_TRY(check_lengths("gen_forward_ragged", lengths_host, B, T_max));
    SVB_CHECK(g, SVB_ERR_INVALID, "gen_forward_ragged: null handle");
    return forward_impl(g, mel_dev, false, f0_dev, rand_ini_dev, noise_dev, seed, B, T_max, wav_dev, as_stream(stream), lengths_host);
}

extern "C" int svb_gen_spec2wav_host(svb_gen_t *g, const float *mel_host, const float *f0_host, uint64_t seed, int32_t B,
                                     int32_t T, float *wav_host, void *stream) {
    SVB_CHECK(g && g->finalized, SVB_ERR_STATE, "spec2wav: generator not finalized");
    SVB_CHECK(mel_host && wav_host && B > 0 && T > 0, SVB_ERR_INVALID, "spec2wav: null buffer or empty input");
    SVB_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = as_stream(stream);
    const size_t n_mel = (size_t)B * T * g->cfg.n_mel, n_f0 = f0_host ? (size_t)B * T : 0;
    const size_t n_in = n_mel + n_f0, n_out = (size_t)B * T * g->hop;
    if (n_in > g->pin_in_cap) {
        if (g->pin_in) cudaFreeHost(g->pin_in);
        if (g->dev_in) cudaFree(g->dev_in);
        g->pin_in = nullptr, g->dev_in = nullptr, g->pin_in_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_in, n_in * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_in, n_in * 4));
        g->pin_in_cap = n_in;
    }
    if (n_out > g->pin_out_cap) {
        if (g->pin_out) cudaFreeHost(g->pin_out);
        if (g->dev_out) cudaFree(g->dev_out);
        g->pin_out = nullptr, g->dev_out = nullptr, g->pin_out_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_out, n_out * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_out, n_out * 4));
        g->pin_out_cap = n_out;
    }
    memcpy(g->pin_in, mel_host, n_mel * 4);
    if (f0_host) memcpy(g->pin_in + n_mel, f0_host, n_f0 * 4);
    SVB_CUDA(cudaMemcpyAsync(g->dev_in, g->pin_in, n_in * 4, cudaMemcpyHostToDevice, st));
    SVB_TRY(forward_impl(g, g->dev_in, true, f0_host ? g->dev_in + n_mel : nullptr, nullptr, nullptr, seed, B, T,
                         g->dev_out, st));
    SVB_CUDA(cudaMemcpyAsync(g->pin_out, g->dev_out, n_out * 4, cudaMemcpyDeviceToHost, st));
    SVB_CUDA(cudaStreamSynchronize(st));
    memcpy(wav_host, g->pin_out, n_out * 4);
    return SVB_OK;
}

// ---- save_wav's sample conversion on the device (utils/audio.py:11-16): [norm: wav / max|wav| per clip,] wav * 32767,
// numpy's float -> int16 cast (truncation toward zero).  Done before the D2H copy, the transfer is 2 bytes per sample.
namespace {
// off [B + 1] (frames, optional): clip b is the packed range [off[b] * hop, off[b + 1] * hop) instead of [b * n, (b + 1) * n)
__global__ void clip_absmax_kernel(const float *__restrict__ x, long long n, unsigned *__restrict__ mx, const int *__restrict__ off, int hop) {
    const int b = blockIdx.y;
    const size_t base = off ? (size_t)off[b] * hop : (size_t)b * n;
    if (off) n = (long long)(off[b + 1] - off[b]) * hop;
    float m = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = fmaxf(m, fabsf(x[base + i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(mx + b, __float_as_uint(m));      // non-negative floats order like their bit patterns
}
__global__ void to_int16_kernel(const float *__restrict__ x, long long n, const unsigned *__restrict__ mx, int16_t *__restrict__ y,
                                const int *__restrict__ off, int hop) {
    const int b = blockIdx.y;
    const size_t base = off ? (size_t)off[b] * hop : (size_t)b * n;
    if (off) n = (long long)(off[b + 1] - off[b]) * hop;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float v = x[base + i];
        if (mx) v = __fdiv_rn(v, __uint_as_float(mx[b]));
        v = __fmul_rn(v, 32767.f);
        y[base + i] = (int16_t)__float2int_rz(v);
    }
}
// n = samples per clip (with `off`: of the longest clip, sizes the grid)
int wav_to_int16(const float *wav_dev, int B, long long n, int norm, int16_t *out_dev, unsigned *mx_dev, cudaStream_t st,
                 const int *off = nullptr, int hop = 1) {
    const dim3 grid((unsigned)std::min<long long>((n + 255) / 256, 148 * 4), (unsigned)B);
    if (norm) {
        SVB_CUDA(cudaMemsetAsync(mx_dev, 0, (size_t)B * sizeof(unsigned), st));
        clip_absmax_kernel<<<grid, 256, 0, st>>>(wav_dev, n, mx_dev, off, hop);
    }
    to_int16_kernel<<<grid, 256, 0, st>>>(wav_dev, n, norm ? mx_dev : nullptr, out_dev, off, hop);
    SVB_CUDA(cudaGetLastError());
    return SVB_OK;
}
}  // namespace

extern "C" int svb_wav_to_int16(const float *wav_dev, int32_t B, int64_t n, int32_t norm, int16_t *out_dev, void *stream) {
    SVB_CHECK(wav_dev && out_dev && B > 0 && n > 0, SVB_ERR_INVALID, "wav_to_int16: bad argument");
    cudaStream_t st = as_stream(stream);
    unsigned *mx = nullptr;
    if (norm) SVB_CUDA(cudaMallocAsync((void **)&mx, (size_t)B * sizeof(unsigned), st));
    const int rc = wav_to_int16(wav_dev, B, n, norm, out_dev, mx, st);
    if (mx) cudaFreeAsync(mx, st);
    return rc;
}

extern "C" int svb_gen_spec2wav_host_i16(svb_gen_t *g, const float *mel_host, const float *f0_host, uint64_t seed, int32_t B,
                                         int32_t T, int32_t norm, int16_t *wav_host, void *stream) {
    SVB_CHECK(g && g->finalized, SVB_ERR_STATE, "spec2wav_i16: generator not finalized");
    SVB_CHECK(mel_host && wav_host && B > 0 && T > 0, SVB_ERR_INVALID, "spec2wav_i16: null buffer or empty input");
    SVB_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = as_stream(stream);
    const size_t n_mel = (size_t)B * T * g->cfg.n_mel, n_f0 = f0_host ? (size_t)B * T : 0;
    const size_t n_in = n_mel + n_f0, n_out = (size_t)B * T * g->hop;
    if (n_in > g->pin_in_cap) {
        if (g->pin_in) cudaFreeHost(g->pin_in);
        if (g->dev_in) cudaFree(g->dev_in);
        g->pin_in = nullptr, g->dev_in = nullptr, g->pin_in_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_in, n_in * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_in, n_in * 4));
        g->pin_in_cap = n_in;
    }
    if (n_out > g->pin_out_cap) {
        if (g->pin_out) cudaFreeHost(g->pin_out);
        if (g->dev_out) cudaFree(g->dev_out);
        g->pin_out = nullptr, g->dev_out = nullptr, g->pin_out_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_out, n_out * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_out, n_out * 4));
        g->pin_out_cap = n_out;
    }
    if (n_out > g->i16_cap) {
        if (g->dev_i16) cudaFree(g->dev_i16);
        g->dev_i16 = nullptr, g->i16_cap = 0;
        SVB_CUDA(cudaMalloc((void **)&g->dev_i16, n_out * 2 + (size_t)4096 * sizeof(unsigned)));
        g->i16_cap = n_out;
    }
    SVB_CHECK(B <= 4096, SVB_ERR_INVALID, "spec2wav_i16: batch %d > 4096", B);
    memcpy(g->pin_in, mel_host, n_mel * 4);
    if (f0_host) memcpy(g->pin_in + n_mel, f0_host, n_f0 * 4);
    SVB_CUDA(cudaMemcpyAsync(g->dev_in, g->pin_in, n_in * 4, cudaMemcpyHostToDevice, st));
    SVB_TRY(forward_impl(g, g->dev_in, true, f0_host ? g->dev_in + n_mel : nullptr, nullptr, nullptr, seed, B, T, g->dev_out, st));
    unsigned *mx;
    mx = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(g->dev_i16) + (g->i16_cap * 2 + 3) / 4 * 4);
    SVB_TRY(wav_to_int16(g->dev_out, B, (long long)T * g->hop, norm, g->dev_i16, mx, st));
    // the pinned float staging buffer is large enough for the 2-byte samples
    SVB_CUDA(cudaMemcpyAsync(g->pin_out, g->dev_i16, n_out * 2, cudaMemcpyDeviceToHost, st));
    SVB_CUDA(cudaStreamSynchronize(st));
    memcpy(wav_host, g->pin_out, n_out * 2);
    return SVB_OK;
}

// ---- spec2wav over a ragged batch from host memory (packed clip after clip, svb_wav2spec_batch_host's convention):
// one H2D of mel + f0, the forward reads the packed rows directly (layout kernel / NSF source) and conv_post writes the packed
// waveform, [int16 conversion with a per-clip peak,] one D2H.
namespace {
int spec2wav_ragged(svb_gen_t *g, const char *what, const float *mel_host, const float *f0_host, const int32_t *lens, int B,
                    uint64_t seed, bool i16, int norm, void *wav_host, void *stream) {
    SVB_CHECK(mel_host && wav_host, SVB_ERR_INVALID, "%s: null buffer", what);
    SVB_TRY(check_lengths(what, lens, B, 0));
    SVB_CHECK(g && g->finalized, SVB_ERR_STATE, "%s: generator not finalized", what);
    SVB_CHECK(!i16 || B <= 4096, SVB_ERR_INVALID, "%s: batch %d > 4096", what, B);
    int T_max = 0;
    size_t frames = 0;
    for (int b = 0; b < B; ++b) T_max = std::max(T_max, (int)lens[b]), frames += lens[b];
    SVB_CUDA(cudaSetDevice(g->device));
    cudaStream_t st = as_stream(stream);
    const size_t n_mel = frames * g->cfg.n_mel, n_f0 = f0_host ? frames : 0;
    const size_t n_in = n_mel + n_f0, n_out = frames * g->hop;
    if (n_in > g->pin_in_cap) {
        if (g->pin_in) cudaFreeHost(g->pin_in);
        if (g->dev_in) cudaFree(g->dev_in);
        g->pin_in = nullptr, g->dev_in = nullptr, g->pin_in_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_in, n_in * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_in, n_in * 4));
        g->pin_in_cap = n_in;
    }
    if (n_out > g->pin_out_cap) {
        if (g->pin_out) cudaFreeHost(g->pin_out);
        if (g->dev_out) cudaFree(g->dev_out);
        g->pin_out = nullptr, g->dev_out = nullptr, g->pin_out_cap = 0;
        SVB_CUDA(cudaMallocHost((void **)&g->pin_out, n_out * 4));
        SVB_CUDA(cudaMalloc((void **)&g->dev_out, n_out * 4));
        g->pin_out_cap = n_out;
    }
    if (i16 && n_out > g->i16_cap) {
        if (g->dev_i16) cudaFree(g->dev_i16);
        g->dev_i16 = nullptr, g->i16_cap = 0;
        SVB_CUDA(cudaMalloc((void **)&g->dev_i16, n_out * 2 + (size_t)4096 * sizeof(unsigned)));
        g->i16_cap = n_out;
    }
    memcpy(g->pin_in, mel_host, n_mel * 4);
    if (f0_host) memcpy(g->pin_in + n_mel, f0_host, n_f0 * 4);
    SVB_CUDA(cudaMemcpyAsync(g->dev_in, g->pin_in, n_in * 4, cudaMemcpyHostToDevice, st));
    SVB_TRY(forward_impl(g, g->dev_in, true, f0_host ? g->dev_in + n_mel : nullptr, nullptr, nullptr, seed, B, T_max, g->dev_out, st,
                         lens, true));
    if (i16) {
        unsigned *mx = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(g->dev_i16) + (g->i16_cap * 2 + 3) / 4 * 4);
        SVB_TRY(wav_to_int16(g->dev_out, B, (long long)T_max * g->hop, norm, g->dev_i16, mx, st, g->rg_dev + 2 * B, g->hop));
        SVB_CUDA(cudaMemcpyAsync(g->pin_out, g->dev_i16, n_out * 2, cudaMemcpyDeviceToHost, st));
    } else {
        SVB_CUDA(cudaMemcpyAsync(g->pin_out, g->dev_out, n_out * 4, cudaMemcpyDeviceToHost, st));
    }
    SVB_CUDA(cudaStreamSynchronize(st));
    memcpy(wav_host, g->pin_out, n_out * (i16 ? 2 : 4));
    return SVB_OK;
}
}  // namespace

extern "C" int svb_gen_spec2wav_ragged_host(svb_gen_t *g, const float *mel_host, const float *f0_host, const int32_t *lengths_host,
                                            int32_t B, uint64_t seed, float *wav_host, void *stream) {
    return spec2wav_ragged(g, "spec2wav_ragged", mel_host, f0_host, lengths_host, B, seed, false, 0, wav_host, stream);
}

extern "C" int svb_gen_spec2wav_ragged_host_i16(svb_gen_t *g, const float *mel_host, const float *f0_host, const int32_t *lengths_host,
                                                int32_t B, uint64_t seed, int32_t norm, int16_t *wav_host, void *stream) {
    return spec2wav_ragged(g, "spec2wav_ragged_i16", mel_host, f0_host, lengths_host, B, seed, true, norm, wav_host, stream);
}

extern "C" int svb_gen_get_tap(svb_gen_t *g, const char *name, float *out_dev, int64_t capacity_floats, int64_t *shape3,
                               void *stream) {
    SVB_CHECK(g && name && out_dev && shape3, SVB_ERR_INVALID, "get_tap: null argument");
    auto it = g->taps.find(name);
    SVB_CHECK(it != g->taps.end(), SVB_ERR_INVALID, "get_tap: no activation named '%s' in the last forward", name);
    const Tap &t = it->second;
    const int B = g->last_B;
    shape3[0] = B, shape3[1] = t.C, shape3[2] = t.T;
    SVB_CHECK((int64_t)B * t.C * t.T <= capacity_floats, SVB_ERR_INVALID, "get_tap: buffer too small");
    cudaStream_t st = as_stream(stream);
    if (t.plain) SVB_CUDA(cudaMemcpyAsync(out_dev, t.p, (size_t)B * t.T * 4, cudaMemcpyDeviceToDevice, st));
    else SVB_TRY(launch_c4t_to_nct(t.p, out_dev, B, t.C, t.T, t.Tp, st));
    return SVB_OK;
}

extern "C" int64_t svb_gen_hop(const svb_gen_t *g) { return g ? g->hop : 0; }
extern "C" int64_t svb_gen_last_launches(const svb_gen_t *g) { return g ? g->last_launches : 0; }
extern "C" double svb_gen_last_flops(const svb_gen_t *g) { return g ? g->last_flops : 0.0; }
extern "C" int svb_gen_enable_timing(svb_gen_t *g, int32_t on) {
    SVB_CHECK(g, SVB_ERR_INVALID, "enable_timing: null handle");
    g->timing = on != 0;
    g->profile = on == 2;
    return SVB_OK;
}
extern "C" int32_t svb_gen_profile_count(svb_gen_t *g) { return g ? (int32_t)g->recs.size() : 0; }
extern "C" int svb_gen_profile_get(svb_gen_t *g, int32_t i, char *name, int32_t name_cap, float *ms, double *bytes,
                                   double *flops) {
    SVB_CHECK(g && i >= 0 && i < (int32_t)g->recs.size() && name && ms && bytes && flops && name_cap > 0, SVB_ERR_INVALID,
              "profile_get: bad argument");
    const auto &r = g->recs[i];
    SVB_CUDA(cudaEventSynchronize(r.e1));
    SVB_CUDA(cudaEventElapsedTime(ms, r.e0, r.e1));
    snprintf(name, name_cap, "%s", r.name);
    *bytes = r.bytes, *flops = r.flops;
    return SVB_OK;
}
extern "C" float svb_gen_last_ms(svb_gen_t *g) {
    if (!g || !g->timing) return -1.f;
    float ms = -1.f;
    if (cudaEventSynchronize(g->ev1) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, g->ev0, g->ev1) != cudaSuccess) return -1.f;
    return ms;
}
