// fused_v46.cu -- hand-scheduled fast path for the rife-v4.6 IFNet (the BASELINE hot path): the ~50 elementwise
// graph nodes between the conv stacks (Interp / Crop / BinaryOp / Eltwise / Concat / rife.Warp / Sigmoid, SURVEY.md
// Appendix B) collapse into three HBM kernels, and every convolution runs on the tcgen05 kernel (tc_conv.cu):
//   head0   x0 = bilinear(cat(I0, I1, T), 1/8)                                   -> C8 space-to-depth, split fp16
//   head<S> U = bilinear(d_{k-1}, S'); F = F + S'*U[0:4] (k = 1: F = S'*U[0:4]); M = M + U[4]   (the update after block k-1)
//           x = cat(bilinear(cat(warp(I0,F01), warp(I1,F23), T, M), 1/S), bilinear(F, 1/S) / S)   (S = 4, 2, 1)
//   tail    F3 = F + d3[0:4]; M3 = M + d3[4]; out = warp(I0,F3_01)*sigmoid(M3) + warp(I1,F3_23)*(1 - sigmoid(M3)) -> u8
// The kernels read the frames as padded RGBX bytes (one launch converts every distinct frame of a batch) and evaluate
// v = u8 * (1/255) on the fly -- exactly what rife_preproc would have stored (src/rife.cpp:4152-4211) -- so the fp32 planar
// copies of the frames (25 MB each at 1080p, gathered 4 x per pair) never exist on this path.
// Arithmetic is the generic executor's, operation for operation (same lin_coeff, H pass then V pass, same warp), so the
// two paths agree to fp32 rounding; Engine::load() additionally checks the fast path against the generic executor on a
// small random frame pair and silently keeps the generic path when the graph is not the expected one.
// Reference dataflow: /root/reference/models/rife-v4.6/flownet.param:1-217.
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <utility>
#include <vector>

#include "fused_v46.h"
#include "kernels.h"
#include "tc_conv.h"

#include "fused_v46_kernels.cuh"

namespace rife {

using namespace fusedk;

namespace {

inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

}  // namespace

// Option "ktime" (or RIFE_B200_KTIME=1): CUDA-event time of every stage of run_batch, recorded on the stream the kernels run
// on.  Diagnostics: the stream is synchronised after each batch, so lanes do not overlap while it is on.
struct StageTimer {
    bool on = false;
    std::vector<cudaEvent_t> ev;
    std::vector<std::string> names;
    std::vector<std::pair<std::string, double>> acc;
    std::vector<int> cnt;
    int batches = 0;
    StageTimer() { const char* e = getenv("RIFE_B200_KTIME"); on = e && atoi(e) != 0; }
    void begin(cudaStream_t st) { if (!on) return; names.clear(); mark(nullptr, st); }
    void mark(const char* name, cudaStream_t st) {
        if (!on) return;
        size_t i = names.size();
        if (ev.size() <= i) { cudaEvent_t e; cudaEventCreate(&e); ev.push_back(e); }
        cudaEventRecord(ev[i], st);
        names.push_back(name ? name : "");
    }
    void end(cudaStream_t st) {
        if (!on) return;
        cudaStreamSynchronize(st);
        for (size_t i = 1; i < names.size(); i++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ev[i - 1], ev[i]);
            size_t j = 0;
            for (; j < acc.size(); j++) if (acc[j].first == names[i]) break;
            if (j == acc.size()) { acc.push_back({names[i], 0.0}); cnt.push_back(0); }
            acc[j].second += ms; cnt[j]++;
        }
        batches++;
    }
    void reset() { acc.clear(); cnt.clear(); batches = 0; }
    // one line per stage: "<name>\t<us per batch>\t<launches per batch>"; first line "batches\t<n>"
    std::string report() const {
        char buf[160];
        snprintf(buf, sizeof buf, "batches\t%d\n", batches);
        std::string r = buf;
        for (size_t j = 0; j < acc.size() && batches; j++) {
            snprintf(buf, sizeof buf, "%s\t%.2f\t%d\n", acc[j].first.c_str(), 1e3 * acc[j].second / batches, cnt[j] / batches);
            r += buf;
        }
        return r;
    }
    ~StageTimer() {
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
        if (!on || !batches || !getenv("RIFE_B200_KTIME")) return;
        double tot = 0;
        for (auto& a : acc) tot += a.second;
        fprintf(stderr, "[rife_b200 ktime] %d batches, %.3f ms per batch\n", batches, tot / batches);
        for (size_t j = 0; j < acc.size(); j++)
            fprintf(stderr, "[rife_b200 ktime] %-22s %8.1f us/batch (%2d launches) %5.1f %%\n", acc[j].first.c_str(), 1e3 * acc[j].second / batches, cnt[j] / batches, 100 * acc[j].second / tot);
    }
};


// sole consumer layer of blob b, or -1
static int consumer_of(const Net& net, int b) {
    int found = -1;
    for (size_t i = 0; i < net.layers.size(); i++)
        for (int bb : net.layers[i].bottoms)
            if (bb == b) { if (found >= 0) return -1; found = (int)i; }
    return found;
}

int V46Runner::init(const Net* net, const NetRunner* weights, std::string& err) {
    ok_ = false;
    net_ = net;
    wr_ = weights;
    conv_.clear();
    for (size_t i = 0; i < net->layers.size(); i++) {
        const Layer& L = net->layers[i];
        if (L.type == "Convolution" || L.type == "Deconvolution") conv_.push_back((int)i);
    }
    if (conv_.size() != 44) { err = "not a 4-block IFNet"; return -1; }
    // rife-v4.6: deconv -> 24 channels -> PixelShuffle(2); rife-v4: deconv -> 5 channels at half the block resolution
    const int head_out = net->layers[conv_[10]].geti(0, 0);
    if (head_out != 24 && head_out != 5) { err = "unexpected flow-head width"; return -1; }
    v4_ = head_out == 5;
    static const int cw[4] = {192, 128, 96, 64};
    for (int k = 0; k < 4; k++) {
        for (int j = 0; j < 11; j++) {
            const int li = conv_[k * 11 + j];
            const Layer& L = net->layers[li];
            const DeviceWeights& W = weights->weights(li);
            bool isdeconv = j == 10;
            if ((L.type == "Deconvolution") != isdeconv || !W.wpk) { err = "layer order / tensor-core eligibility mismatch at " + L.name; return -1; }
            int cout = L.geti(0, 0);
            int want = j == 0 ? cw[k] / 2 : (j == 10 ? head_out : cw[k]);
            int wcin = j == 0 ? (k == 0 ? 7 : 12) : (j == 1 ? cw[k] / 2 : cw[k]);
            if (cout != want || W.cin != wcin || (j < 2) != (W.tc_s2 != 0)) { err = "unexpected shape at " + L.name; return -1; }
            ConvCfg& c = cfg_[k * 11 + j];
            c = ConvCfg();
            c.layer = li;
            if (isdeconv) continue;
            // activation: the convolution's own fused leaky (v4.6 stride-2 convs), or the layer(s) that consume its output:
            // PReLU (v4, every conv) / BinaryOp add + ReLU (v4.6 residual convs: y = leaky(conv(y) + y))
            if (L.geti(9, 0) == 2) {
                const ParamVal* ap = L.get(10);
                c.act_mode = 1;
                c.slope = ap && !ap->af.empty() ? ap->af[0] : 0.f;
                continue;
            }
            int c1 = L.tops.empty() ? -1 : consumer_of(*net, L.tops[0]);
            if (c1 >= 0 && net->layers[c1].type == "PReLU") {
                const Layer& A = net->layers[c1];
                if (A.slope.size() == 1) { c.act_mode = 1; c.slope = A.slope[0]; }
                else if ((int)A.slope.size() == cout && weights->weights(c1).slope) { c.act_mode = 2; c.prelu = weights->weights(c1).slope; }
                else { err = "unexpected PReLU form after " + L.name; return -1; }
                if (j == 9) {  // v4: one residual around the eight convolutions, added after the last PReLU (BinaryOp add_0 ...)
                    int c2 = A.tops.empty() ? -1 : consumer_of(*net, A.tops[0]);
                    if (c2 < 0 || net->layers[c2].type != "BinaryOp" || net->layers[c2].geti(0, 0) != 0 || net->layers[c2].bottoms.size() != 2) { err = "no residual add after " + A.name; return -1; }
                    c.res_mode = 2;
                }
            } else if (c1 >= 0 && j >= 2 && net->layers[c1].type == "BinaryOp" && net->layers[c1].geti(0, 0) == 0 && net->layers[c1].bottoms.size() == 2) {
                int c2 = net->layers[c1].tops.empty() ? -1 : consumer_of(*net, net->layers[c1].tops[0]);
                if (c2 < 0 || net->layers[c2].type != "ReLU") { err = "no activation after the residual add of " + L.name; return -1; }
                c.act_mode = 1;
                c.slope = net->layers[c2].getf(0, 0.f);
                c.res_mode = 1;
            } else { err = "unexpected consumer of " + L.name; return -1; }
        }
        // the two layouts this runner schedules: v4.6 = residual on every chain conv, v4 = on the last one only
        for (int j = 2; j < 10; j++) {
            const int want = v4_ ? (j == 9 ? 2 : 0) : 1;
            if (cfg_[k * 11 + j].res_mode != want) { err = "unexpected residual structure in block " + std::to_string(k); return -1; }
        }
    }
    if (net->find_blob("flow3") < 0 || net->find_blob("out0") < 0) { err = "no flow3 / out0 in graph"; return -1; }
    // option "head_pack": the first stride-2 conv of blocks 1-3 reads a 16-slot tensor whose slots 12..15 carry the lo parts
    // of the flow channels 8..11 -- its weights for those slots are copies of the flow channels' weights
    for (int k = 0; k < 4; k++) {
        if (wpk_head_[k]) { cudaFree(wpk_head_[k]); wpk_head_[k] = nullptr; }
        if (k == 0) continue;  // 7 channels, no flow input: the plain hi plane is all there is
        const Layer& L = net->layers[cfg_[k * 11].layer];
        const int cout = L.geti(0, 0), cin = 12;
        std::vector<float> w16((size_t)cout * 16 * 9, 0.f);
        for (int oc = 0; oc < cout; oc++)
            for (int ic = 0; ic < 16; ic++)
                for (int t = 0; t < 9; t++) w16[((size_t)oc * 16 + ic) * 9 + t] = L.weight[((size_t)oc * cin + (ic < 12 ? ic : ic - 4)) * 9 + t];
        std::vector<uint16_t> pk;
        pack_conv3x3s2_weights(w16.data(), cout, 16, 16, weights->weights(cfg_[k * 11].layer).tcN, pk);
        if (cudaMalloc(&wpk_head_[k], pk.size() * 2) != cudaSuccess) { err = "cudaMalloc failed"; return -2; }
        cudaMemcpy(wpk_head_[k], pk.data(), pk.size() * 2, cudaMemcpyHostToDevice);
    }
    ok_ = true;
    return 0;
}

V46Runner::~V46Runner() {
    for (void* p : bufs_) cudaFree(p);
    for (auto& p : wpk_head_) cudaFree(p);
    delete tm_;
}

void V46Runner::set_ktime(int on) {
    if (!tm_) tm_ = new StageTimer();
    tm_->on = on != 0;
    tm_->reset();
}
std::string V46Runner::stage_report() const { return tm_ ? tm_->report() : std::string("batches\t0\n"); }

int V46Runner::ensure(int w, int h, int batch, std::string& err) {
    const int wp = (w + 31) / 32 * 32, hp = (h + 31) / 32 * 32;
    if (wp == wp_ && hp == hp_ && batch <= cap_) return 0;
    const size_t B = (size_t)batch;
    for (void* p : bufs_) cudaFree(p);
    bufs_.clear();
    auto alloc = [&](size_t bytes) -> void* {
        void* p = nullptr;
        if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
        bufs_.push_back(p);
        return p;
    };
    const size_t plane = (size_t)wp * hp;
    rgbx_ = (uchar4*)alloc(2 * B * plane * 4);
    F_ = (float*)alloc(B * 4 * plane * 4);
    M_ = (float*)alloc(B * plane * 4);
    static const int S[4] = {8, 4, 2, 1};
    bool fail = !F_ || !M_ || !rgbx_;
    for (int k = 0; k < 4; k++) {
        const size_t hk = hp / S[k], wk = wp / S[k];
        static const int cw[4] = {192, 128, 96, 64};
        d_[k] = (float*)alloc(B * 6 * hk * wk * 4);                                // v4.6: 6 planes at the block resolution; v4: 5 at half of it
        x_[k] = (__half*)alloc(B * 16 * hk * wk * 2 * 2);                         // head, C8 s2d, hi+lo
        y0_[k] = (__half*)alloc(B * (cw[k] / 2) * (hk / 2) * (wk / 2) * 2 * 2);   // conv0 out, C8 s2d
        a_[k] = (__half*)alloc(B * cw[k] * (hk / 4) * (wk / 4) * 2 * 2);          // residual chain ping
        b_[k] = (__half*)alloc(B * cw[k] * (hk / 4) * (wk / 4) * 2 * 2);          // residual chain pong
        c_[k] = v4_ ? (__half*)alloc(B * cw[k] * (hk / 4) * (wk / 4) * 2 * 2) : nullptr;  // v4: conv1's output stays live as the chain's residual
        fail = fail || !d_[k] || !x_[k] || !y0_[k] || !a_[k] || !b_[k] || (v4_ && !c_[k]);
    }
    if (fail) { err = "cudaMalloc failed"; wp_ = hp_ = 0; cap_ = 0; return -2; }
    wp_ = wp;
    hp_ = hp;
    cap_ = batch;
    return 0;
}

int V46Runner::conv(int slot, const __half* in, __half* out, const __half* res, float* out_f32, int oh, int ow, bool out_s2d, int batch, bool split_in,
                    bool split_out, cudaStream_t st) {
    const ConvCfg& c = cfg_[slot];
    const int li = c.layer;
    const Layer& L = net_->layers[li];
    const DeviceWeights& W = wr_->weights(li);
    TcConvArgs a;
    memset(&a, 0, sizeof a);
    a.wpk = (const __half*)W.wpk;
    if (head_pack_ && slot % 11 == 0 && wpk_head_[slot / 11]) a.wpk = wpk_head_[slot / 11];  // flow channels seen twice (hi + lo slots)
    a.bias = W.biasN;
    a.H = oh; a.W = ow; a.Cin = W.cinp; a.Cout = L.geti(0, 0); a.N = W.tcN;
    a.split_in = split_in;
    a.s2 = W.tc_s2;
    a.num_sms = wr_->num_sms;
    a.batch = batch;
    a.in_bstride = (size_t)(W.tc_s2 ? 4 : 1) * W.cinp * oh * ow * 2;  // room for hi + lo planes of one image (also when only hi is used)
    if (L.type == "Convolution") {
        a.out_bstride = a.res_bstride = (size_t)L.geti(0, 0) * oh * ow * 2;
        a.epi = TC_EPI_C8;
        a.out = out;
        a.out_plane = (size_t)a.Cout * oh * ow;
        a.split_out = split_out;
        a.out_s2d = out_s2d;
        a.act_mode = c.act_mode;
        a.slope = c.slope;
        a.prelu = c.prelu;
        if (res && c.res_mode) { a.res = res; a.res_plane = a.out_plane; a.res_split = res_split_; a.res_mode = c.res_mode; }
    } else if (!v4_) {
        a.epi = TC_EPI_DECONV;
        a.out_f32 = out_f32;
        a.ocs = W.ocs;
        a.ps = 2;
        a.out_planes = 5;  // flow (4) + mask (1); the 6th PixelShuffle plane is never read by head / tail
        a.outf_bstride = (size_t)6 * (oh * 4) * (ow * 4);
    } else {
        a.epi = TC_EPI_DECONV;  // 5 channels, no PixelShuffle: planar fp32 [5][2*oh][2*ow]
        a.out_f32 = out_f32;
        a.ocs = W.ocs;
        a.ps = 1;
        a.outf_bstride = (size_t)5 * (oh * 2) * (ow * 2);
    }
    return launch_tc_conv(a, in, st);
}

int V46Runner::run(const uint8_t* d_in0, const uint8_t* d_in1, int w, int h, float t, uint8_t* d_out, cudaStream_t st, std::string& err) {
    return run_batch(1, &d_in0, &d_in1, w, h, &t, &d_out, st, err);
}

// n <= V46_MAX_BATCH pairs in lock-step: every kernel covers all n images (blockIdx.z / the image-major tile index of the
// conv), so the latency-bound small blocks (17-136 CTAs per image at 1080p) fill the machine.
int V46Runner::run_batch(int n, const uint8_t* const* d_in0, const uint8_t* const* d_in1, int w, int h, const float* ts, uint8_t* const* d_out,
                         cudaStream_t st, std::string& err) {
    if (!ok_) { err = "fast path not initialised"; return -1; }
    if (n < 1 || n > V46_MAX_BATCH) { err = "bad batch size"; return -1; }
    if (ensure(w, h, n, err)) return -2;
    const int wp = wp_, hp = hp_;
    const size_t plane = (size_t)wp * hp;
    static const int S[4] = {8, 4, 2, 1};
    TBatch tb;
    OutBatch ob;
    InBatch ib;
    SrcBatch sb;
    int nu = 0;  // distinct frames of this batch: the second frame of pair i is usually the first frame of pair i + 1
    auto slot = [&](const uint8_t* p) {
        for (int i = 0; i < nu; i++) if (sb.p[i] == p) return i;
        sb.p[nu] = p;
        return nu++;
    };
    for (int b = 0; b < V46_MAX_BATCH; b++) {
        tb.t[b] = b < n ? ts[b] : 0.f;
        ob.p[b] = b < n ? d_out[b] : nullptr;
        ib.p0[b] = b < n ? rgbx_ + (size_t)slot(d_in0[b]) * plane : nullptr;
        ib.p1[b] = b < n ? rgbx_ + (size_t)slot(d_in1[b]) * plane : nullptr;
    }
    for (int i = nu; i < 2 * V46_MAX_BATCH; i++) sb.p[i] = nullptr;
    // recompute_fm: 0 = F / M live in memory between block 2's head and the tail; 1 = the head of block 3 stops storing them
    // (the tail redoes the block-2 update); 2 = they are never stored at all (heads 2, 3 and the tail rebuild them from d0..d2)
    // (rife-v4.6 layout only; measured slower than storing, profiles/README.md)
    const bool rc2 = !v4_ && recompute_ >= 2, rc1 = !v4_ && recompute_ == 1;
    const int dch = v4_ ? 5 : 6;  // planes of the block outputs d_k (v4: at half the block resolution)
    if (!tm_) tm_ = new StageTimer();
    StageTimer& tm = *tm_;
    tm.begin(st);
    bool vec = (w & 3) == 0;
    for (int i = 0; i < nu; i++) vec = vec && ((uintptr_t)sb.p[i] & 3) == 0;
    if (vec) rgbx4_kernel<<<dim3(cdiv(wp / 4, 128), hp, nu), 128, 0, st>>>(sb, w, h, wp, hp, rgbx_, bgr_);
    else rgbx_kernel<<<dim3(cdiv(wp, 128), hp, nu), 128, 0, st>>>(sb, w, h, wp, hp, rgbx_, bgr_);
    g_launch_count++;
    tm.mark("rgbx", st);
    char nm[32];
    for (int k = 0; k < 4; k++) {
        const int hk = hp / S[k], wk = wp / S[k];
        dim3 g(cdiv(wk, 128), hk, n);
        // head of block k, fused with the flow / mask update that follows block k-1
        if (k == 0) head0_kernel<<<g, 128, 0, st>>>(ib, tb, hp, wp, hk, wk, x_[0], head_pack_);
        else if (v4_) {
            // rife-v4: d_{k-1} has 5 planes at 1/(2*S_{k-1}) of the frame, so the up-sampling factors double
            if (k == 1) head_update_kernel<4, 16, 0, 16, false><<<g, 128, 0, st>>>(ib, F_, M_, d_[0], hp / 16, wp / 16, nullptr, 0, 0, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[1], dch, head_pack_);
            else if (k == 2) head_update_kernel<2, 8, 1, 16, true><<<g, 128, 0, st>>>(ib, F_, M_, d_[1], hp / 8, wp / 8, d_[0], hp / 16, wp / 16, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[2], dch, head_pack_);
            else head_update_kernel<1, 4, 2, 16, true><<<g, 128, 0, st>>>(ib, F_, M_, d_[2], hp / 4, wp / 4, nullptr, 0, 0, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[3], dch, head_pack_);
        } else if (k == 1) head_update_kernel<4, 8, 0, 8, false><<<g, 128, 0, st>>>(ib, F_, M_, d_[0], hp / 8, wp / 8, nullptr, 0, 0, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[1], dch, head_pack_);
        else if (k == 2) {
            if (rc2) head_update_kernel<2, 4, 1, 8, false><<<g, 128, 0, st>>>(ib, F_, M_, d_[1], hp / 4, wp / 4, d_[0], hp / 8, wp / 8, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[2], dch, head_pack_);
            else head_update_kernel<2, 4, 1, 8, true><<<g, 128, 0, st>>>(ib, F_, M_, d_[1], hp / 4, wp / 4, d_[0], hp / 8, wp / 8, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[2], dch, head_pack_);
        } else {
            if (rc2) head_update_kernel<1, 2, 3, 4, false><<<g, 128, 0, st>>>(ib, F_, M_, d_[2], hp / 2, wp / 2, d_[1], hp / 4, wp / 4, d_[0], hp / 8, wp / 8, tb, hp, wp, hk, wk, x_[3], dch, head_pack_);
            else if (rc1) head_update_kernel<1, 2, 2, 8, false><<<g, 128, 0, st>>>(ib, F_, M_, d_[2], hp / 2, wp / 2, nullptr, 0, 0, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[3], dch, head_pack_);
            else head_update_kernel<1, 2, 2, 8, true><<<g, 128, 0, st>>>(ib, F_, M_, d_[2], hp / 2, wp / 2, nullptr, 0, 0, nullptr, 0, 0, tb, hp, wp, hk, wk, x_[3], dch, head_pack_);
        }
        g_launch_count++;
        snprintf(nm, sizeof nm, "b%d head", k); tm.mark(nm, st);
        const int L0 = k * 11;  // first of the block's 11 convolution slots (cfg_)
        // precision: the block-head tensor and the two stride-2 convs that follow it always run on split (fp32-equivalent)
        // operands -- measured: making conv0's output / conv1's input plain fp16 doubles the 1-LSB flips and, with all four
        // blocks plain, produces 4-LSB errors on the README frames; the residual chain and the deconv of a block are split
        // unless the block is listed in plain_mask_ (plain fp16 activations there)
        const bool sp = !((plain_mask_ >> k) & 1);
        const bool hsp = !((plain_mask_ >> (4 + k)) & 1);  // experimental: read only the hi plane of the head tensor
        int r = conv(L0, x_[k], y0_[k], nullptr, nullptr, hk / 2, wk / 2, true, n, hsp && !head_pack_, true, st);    // 3x3 s2 + activation
        snprintf(nm, sizeof nm, "b%d conv0", k); tm.mark(nm, st);
        __half* y1 = v4_ ? c_[k] : a_[k];
        r |= conv(L0 + 1, y0_[k], y1, nullptr, nullptr, hk / 4, wk / 4, false, n, true, sp, st);         // 3x3 s2 + activation
        snprintf(nm, sizeof nm, "b%d conv1", k); tm.mark(nm, st);
        __half* cur = y1;
        __half* nxt = v4_ ? a_[k] : b_[k];
        res_split_ = sp;
        for (int j = 0; j < 8; j++) {
            // v4.6: y = leaky(conv(y) + y) eight times; v4: y = prelu(conv(y)) eight times, then + conv1's output
            r |= conv(L0 + 2 + j, cur, nxt, v4_ ? y1 : cur, nullptr, hk / 4, wk / 4, false, n, sp, sp, st);
            if (v4_) { cur = nxt; nxt = nxt == a_[k] ? b_[k] : a_[k]; }
            else { __half* tmp = cur; cur = nxt; nxt = tmp; }
        }
        snprintf(nm, sizeof nm, "b%d res x8", k); tm.mark(nm, st);
        r |= conv(L0 + 10, cur, nullptr, nullptr, d_[k], hk / 4, wk / 4, false, n, sp, false, st);        // deconv (+ PixelShuffle) -> flow<k>
        snprintf(nm, sizeof nm, "b%d deconv", k); tm.mark(nm, st);
        if (r) { err = "tensor-core conv launch failed in block " + std::to_string(k); return -3; }
    }
    {
        DSrc ds;
        ds.d[0] = d_[0]; ds.d[1] = d_[1]; ds.d[2] = d_[2];
        const dim3 tg(cdiv(w, 128), h, n);
        if (v4_) tail_kernel<0, 2><<<tg, 128, 0, st>>>(ib, F_, M_, d_[3], hp, wp, ob, w, h, ds, crop_quirk_, dch, bgr_);
        else if (rc2) tail_kernel<2, 1><<<tg, 128, 0, st>>>(ib, F_, M_, d_[3], hp, wp, ob, w, h, ds, crop_quirk_, dch, bgr_);
        else if (rc1) tail_kernel<1, 1><<<tg, 128, 0, st>>>(ib, F_, M_, d_[3], hp, wp, ob, w, h, ds, crop_quirk_, dch, bgr_);
        else tail_kernel<0, 1><<<tg, 128, 0, st>>>(ib, F_, M_, d_[3], hp, wp, ob, w, h, ds, crop_quirk_, dch, bgr_);
    }
    g_launch_count++;
    tm.mark("tail", st);
    tm.end(st);
    return 0;
}

}  // namespace rife
