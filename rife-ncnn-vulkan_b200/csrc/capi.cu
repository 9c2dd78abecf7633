// capi.cu -- the C ABI declared in include/rife_b200.h (thin shell over rife::Engine; catches everything).
#include <new>
#include <string>

#include "../../include/rife_b200.h"
#include "engine.h"
#include "kernels.h"

struct rife_b200 {
    rife::Engine* eng;
    std::string err;
};

#define GUARD_BEGIN try {
#define GUARD_END                                   \
    }                                               \
    catch (const std::bad_alloc&) {                 \
        return RIFE_B200_ERR_INTERNAL;              \
    }                                               \
    catch (...) {                                   \
        return RIFE_B200_ERR_INTERNAL;              \
    }

static int map_err(int r) {
    switch (r) {
        case 0: return RIFE_B200_OK;
        case -1: return RIFE_B200_ERR_ARG;
        case -2: return RIFE_B200_ERR_DEVICE;
        case -3: return RIFE_B200_ERR_MODEL;
        case -4: return RIFE_B200_ERR_STATE;
        default: return RIFE_B200_ERR_INTERNAL;
    }
}

extern "C" {

int rife_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int rife_b200_create(rife_b200_t** handle, int gpuid, int tta_mode, int tta_temporal_mode, int uhd_mode, int /*num_threads*/, int rife_v2, int rife_v4) {
    GUARD_BEGIN
    if (!handle) return RIFE_B200_ERR_ARG;
    *handle = nullptr;
    if (gpuid < 0) return RIFE_B200_ERR_ARG;  // -1 = the reference's CPU mode: rejected by design
    rife_b200* h = new rife_b200();
    h->eng = new rife::Engine(gpuid, tta_mode != 0, tta_temporal_mode != 0, uhd_mode != 0, rife_v2 != 0, rife_v4 != 0);
    int r = h->eng->init();
    if (r) {
        delete h->eng;
        delete h;
        return map_err(r);
    }
    *handle = h;
    return RIFE_B200_OK;
    GUARD_END
}

int rife_b200_load(rife_b200_t* h, const char* modeldir) {
    GUARD_BEGIN
    if (!h || !modeldir) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->load(modeldir));
    GUARD_END
}

int rife_b200_process(rife_b200_t* h, const unsigned char* in0, const unsigned char* in1, int w, int hh, float t, unsigned char* out) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->process_host(in0, in1, w, hh, t, out));
    GUARD_END
}

int rife_b200_process_device(rife_b200_t* h, const unsigned char* in0, const unsigned char* in1, int w, int hh, float t, unsigned char* out) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->process_device(in0, in1, w, hh, t, out));
    GUARD_END
}

int rife_b200_process_batch(rife_b200_t* h, int n, const unsigned char* const* in0, const unsigned char* const* in1, int w, int hh, const float* ts,
                            unsigned char* const* out) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->process_batch(n, in0, in1, w, hh, ts, out));
    GUARD_END
}

int rife_b200_process_batch_device(rife_b200_t* h, int n, const unsigned char* const* in0, const unsigned char* const* in1, int w, int hh, const float* ts,
                                   unsigned char* const* out) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->process_batch_device(n, in0, in1, w, hh, ts, out));
    GUARD_END
}

int rife_b200_set_option(rife_b200_t* h, const char* key, int value) {
    GUARD_BEGIN
    if (!h || !key) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->set_option(key, value));
    GUARD_END
}

int rife_b200_get_option(rife_b200_t* h, const char* key, int* value) {
    GUARD_BEGIN
    if (!h || !key || !value) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->get_option(key, value));
    GUARD_END
}

int rife_b200_weights_size(rife_b200_t* h, size_t* bytes) {
    GUARD_BEGIN
    if (!h || !bytes) return RIFE_B200_ERR_ARG;
    if (h->eng->packed().empty()) return RIFE_B200_ERR_STATE;
    *bytes = h->eng->packed().size();
    return RIFE_B200_OK;
    GUARD_END
}

int rife_b200_weights_export(rife_b200_t* h, void* dst, size_t bytes) {
    GUARD_BEGIN
    if (!h || !dst) return RIFE_B200_ERR_ARG;
    const std::string p = h->eng->packed();
    if (p.empty()) return RIFE_B200_ERR_STATE;
    if (bytes < p.size()) return RIFE_B200_ERR_ARG;
    memcpy(dst, p.data(), p.size());
    return RIFE_B200_OK;
    GUARD_END
}

int rife_b200_load_packed(rife_b200_t* h, const void* src, size_t bytes) {
    GUARD_BEGIN
    if (!h || !src) return RIFE_B200_ERR_ARG;
    return map_err(h->eng->load_packed(src, bytes));
    GUARD_END
}

unsigned long long rife_b200_launch_count(void) { return rife::g_launch_count; }
unsigned long long rife_b200_h2d_bytes(void) { return rife::g_h2d_bytes; }
unsigned long long rife_b200_d2h_bytes(void) { return rife::g_d2h_bytes; }

// the message is copied into a per-thread buffer: several threads may use (and fail on) one handle concurrently
const char* rife_b200_last_error(rife_b200_t* h) {
    static thread_local std::string buf;
    if (!h) return "null handle";
    try { buf = h->eng->last_error(); } catch (...) { return "out of memory"; }
    return buf.c_str();
}

int rife_b200_stage_report(rife_b200_t* h, char* buf, size_t cap) {
    GUARD_BEGIN
    if (!h || !buf || cap == 0) return RIFE_B200_ERR_ARG;
    const std::string r = h->eng->stage_report();
    snprintf(buf, cap, "%s", r.c_str());
    return RIFE_B200_OK;
    GUARD_END
}

int rife_b200_forget_frames(rife_b200_t* h) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    h->eng->forget_frames();
    return RIFE_B200_OK;
    GUARD_END
}

// RIFE::load(const std::wstring&) of the reference's Windows build (src/rife.cpp:80-110): the path is converted to UTF-8
int rife_b200_load_w(rife_b200_t* h, const wchar_t* modeldir) {
    GUARD_BEGIN
    if (!h || !modeldir) return RIFE_B200_ERR_ARG;
    std::string u8;
    for (const wchar_t* p = modeldir; *p; p++) {
        uint32_t c = (uint32_t)*p;
        if (sizeof(wchar_t) == 2 && c >= 0xD800 && c <= 0xDBFF && p[1] >= 0xDC00 && p[1] <= 0xDFFF) { c = 0x10000 + ((c - 0xD800) << 10) + ((uint32_t)p[1] - 0xDC00); p++; }
        if (c < 0x80) u8 += (char)c;
        else if (c < 0x800) { u8 += (char)(0xC0 | (c >> 6)); u8 += (char)(0x80 | (c & 0x3F)); }
        else if (c < 0x10000) { u8 += (char)(0xE0 | (c >> 12)); u8 += (char)(0x80 | ((c >> 6) & 0x3F)); u8 += (char)(0x80 | (c & 0x3F)); }
        else { u8 += (char)(0xF0 | (c >> 18)); u8 += (char)(0x80 | ((c >> 12) & 0x3F)); u8 += (char)(0x80 | ((c >> 6) & 0x3F)); u8 += (char)(0x80 | (c & 0x3F)); }
    }
    return map_err(h->eng->load(u8));
    GUARD_END
}

void rife_b200_destroy(rife_b200_t* h) {
    if (!h) return;
    try {
        delete h->eng;
        delete h;
    } catch (...) {
    }
}

}  // extern "C"

// ---- diagnostics ---------------------------------------------------------------------------------------------
#include <vector>

#include "tc_conv.h"

// mode 2: conv3x3 stride 2 pad 1 (+bias +leaky): in [cin][h][w] (h, w even) -> out [cout][h/2][w/2]
static int selftest_conv_s2(int gpuid, int cin, int cout, int h, int w, int split, const float* in, const float* weight, const float* bias, float slope,
                            float* out_tc, float* out_ref) {
    using namespace rife;
    if ((h | w) & 1 || cout % 16) return RIFE_B200_ERR_ARG;
    if (cudaSetDevice(gpuid) != cudaSuccess) return RIFE_B200_ERR_DEVICE;
    cudaStream_t st = 0;
    const int oh = h / 2, ow = w / 2, cinp = (cin + 15) / 16 * 16;
    const size_t hw = (size_t)h * w, ohw = (size_t)oh * ow;
    std::vector<float> wq((size_t)cout * cin * 9);
    for (size_t i = 0; i < wq.size(); i++) wq[i] = __half2float(__float2half_rn(weight[i]));
    std::vector<uint16_t> wpk;
    pack_conv3x3s2_weights(wq.data(), cout, cin, cinp, cout, wpk);
    int ocpad = (cout + 63) / 64 * 64;
    std::vector<float> t((size_t)cin * 9 * ocpad, 0.f);
    for (int oc = 0; oc < cout; oc++) for (int ic = 0; ic < cin; ic++) for (int k = 0; k < 9; k++) t[((size_t)ic * 9 + k) * ocpad + oc] = wq[((size_t)oc * cin + ic) * 9 + k];
    float *d_in = 0, *d_bias = 0, *d_out_tc = 0, *d_out_ref = 0, *d_wT = 0;
    __half *d_in8 = 0, *d_out8 = 0, *d_wpk = 0;
    cudaMalloc(&d_in, cin * hw * 4); cudaMalloc(&d_in8, (size_t)cinp * hw * 4); cudaMalloc(&d_bias, cout * 4);
    cudaMalloc(&d_out_tc, cout * ohw * 4); cudaMalloc(&d_out_ref, cout * ohw * 4); cudaMalloc(&d_out8, cout * ohw * 4);
    cudaMalloc(&d_wpk, wpk.size() * 2); cudaMalloc(&d_wT, t.size() * 4);
    cudaMemcpy(d_in, in, cin * hw * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_bias, bias, cout * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_wpk, wpk.data(), wpk.size() * 2, cudaMemcpyHostToDevice);
    cudaMemcpy(d_wT, t.data(), t.size() * 4, cudaMemcpyHostToDevice);
    launch_planar_to_c8(d_in, d_in8, cin, h, w, split, st, cinp, 1);
    launch_c8_to_planar(d_in8, d_in, cin, h, w, split, st, cinp, 1);  // reference sees the same (rounded) operand values
    TcConvArgs a;
    memset(&a, 0, sizeof a);
    a.wpk = d_wpk; a.bias = d_bias; a.out = d_out8; a.out_plane = (size_t)cout * ohw; a.slope = slope;
    a.H = oh; a.W = ow; a.Cin = cinp; a.Cout = cout; a.N = cout; a.split_in = split; a.split_out = split; a.epi = TC_EPI_C8; a.act_mode = 1; a.s2 = 1;
    int r = launch_tc_conv(a, d_in8, st);
    if (r) { fprintf(stderr, "launch_tc_conv(s2) failed: %d\n", r); return RIFE_B200_ERR_INTERNAL; }
    launch_c8_to_planar(d_out8, d_out_tc, cout, oh, ow, split, st);
    ConvArgs c;
    memset(&c, 0, sizeof c);
    c.in = d_in; c.wT = d_wT; c.bias = d_bias; c.out = d_out_ref; c.Cin = cin; c.H = h; c.W = w; c.Cout = cout; c.ocpad = ocpad;
    c.OH = oh; c.OW = ow; c.DH = oh; c.DW = ow; c.in_off_y = c.in_off_x = -1; c.out_mul = 1; c.nparity = 1; c.act = 2; c.act_p0 = slope;
    launch_conv(c, 3, 2, st);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { fprintf(stderr, "selftest_conv_s2: %s\n", cudaGetErrorString(e)); return RIFE_B200_ERR_DEVICE; }
    cudaMemcpy(out_tc, d_out_tc, cout * ohw * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(out_ref, d_out_ref, cout * ohw * 4, cudaMemcpyDeviceToHost);
    cudaFree(d_in); cudaFree(d_bias); cudaFree(d_out_tc); cudaFree(d_out_ref); cudaFree(d_wT); cudaFree(d_in8); cudaFree(d_out8); cudaFree(d_wpk);
    return RIFE_B200_OK;
}

extern "C" int rife_b200_selftest_conv(int gpuid, int mode, int cin, int cout, int h, int w, int split, int ps, const float* in, const float* weight,
                                       const float* bias, const float* res, float slope, float* out_tc, float* out_ref) {
    GUARD_BEGIN
    using namespace rife;
    if (!in || !weight || !bias || !out_tc || !out_ref || cin <= 0 || cout <= 0 || h <= 0 || w <= 0) return RIFE_B200_ERR_ARG;
    // mode 3 = mode 1 restricted to the first five PixelShuffle planes (the IFNet flow head: the launcher's out_planes = 5)
    const bool planes5 = mode == 3;
    if (planes5) { if (ps != 2 || cout != 24) return RIFE_B200_ERR_ARG; mode = 1; }
    if (mode != 2 && cin % 16) return RIFE_B200_ERR_ARG;
    if (mode == 2) return selftest_conv_s2(gpuid, cin, cout, h, w, split, in, weight, bias, slope, out_tc, out_ref);
    if (cudaSetDevice(gpuid) != cudaSuccess) return RIFE_B200_ERR_DEVICE;
    cudaStream_t st = 0;
    const size_t hw = (size_t)h * w;
    const int kk = mode == 0 ? 9 : (mode == 4 ? 25 : 16);
    // fp16-exact weights, as in the model files
    std::vector<float> wq((size_t)cout * cin * kk);
    for (size_t i = 0; i < wq.size(); i++) wq[i] = __half2float(__float2half_rn(weight[i]));
    int N, ocs = 0;
    std::vector<uint16_t> wpk;
    if (mode == 0 || mode == 4) {
        N = (cout + 15) / 16 * 16;
        if (N != cout) return RIFE_B200_ERR_ARG;
        if (mode == 0) pack_conv3x3_weights(wq.data(), cout, cin, N, wpk);
        else pack_conv5x5_weights(wq.data(), cout, cin, N, wpk);
    } else {
        ocs = (cout + 7) / 8 * 8;
        N = 4 * ocs;
        pack_deconv4x4_weights(wq.data(), cout, cin, ocs, N, wpk);
    }
    std::vector<float> biasN(N, 0.f);
    if (mode == 0 || mode == 4) for (int i = 0; i < cout; i++) biasN[i] = bias[i];
    else for (int p = 0; p < 4; p++) for (int i = 0; i < cout; i++) biasN[p * ocs + i] = bias[i];
    float *d_in = 0, *d_res = 0, *d_bias = 0, *d_biasN = 0, *d_out_tc = 0, *d_out_ref = 0, *d_wT = 0, *d_tmp = 0;
    __half *d_in8 = 0, *d_res8 = 0, *d_out8 = 0, *d_wpk = 0;
    const size_t out_elems = (mode == 0 || mode == 4) ? (size_t)cout * hw : (size_t)cout * hw * 4;
    cudaMalloc(&d_in, cin * hw * 4); cudaMalloc(&d_in8, cin * hw * 2 * 2); cudaMalloc(&d_bias, cout * 4); cudaMalloc(&d_biasN, N * 4);
    cudaMalloc(&d_out_tc, out_elems * 4); cudaMalloc(&d_out_ref, out_elems * 4); cudaMalloc(&d_tmp, out_elems * 4);
    cudaMalloc(&d_out8, (size_t)cout * hw * 2 * 2); cudaMalloc(&d_wpk, wpk.size() * 2);
    cudaMemcpy(d_in, in, cin * hw * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_bias, bias, cout * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_biasN, biasN.data(), N * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(d_wpk, wpk.data(), wpk.size() * 2, cudaMemcpyHostToDevice);
    cudaMemset(d_out_tc, 0, out_elems * 4);
    const bool self_res = res == in && cin == cout && mode == 0;  // residual = the conv's own input (identity-tap path of the kernel)
    if (res && !self_res) {
        cudaMalloc(&d_res, cout * hw * 4); cudaMalloc(&d_res8, (size_t)cout * hw * 2 * 2);
        cudaMemcpy(d_res, res, cout * hw * 4, cudaMemcpyHostToDevice);
        launch_planar_to_c8(d_res, d_res8, cout, h, w, split, st);
    }
    launch_planar_to_c8(d_in, d_in8, cin, h, w, split, st);
    // the reference result uses exactly the values the tensor path sees (hi+lo reconstruction of the input)
    launch_c8_to_planar(d_in8, d_in, cin, h, w, split, st);
    if (res && !self_res) launch_c8_to_planar(d_res8, d_res, cout, h, w, split, st);
    TcConvArgs a;
    memset(&a, 0, sizeof a);
    a.wpk = d_wpk; a.bias = d_biasN; a.res = self_res ? d_in8 : d_res8; a.res_plane = (size_t)cout * hw; a.res_split = split;
    a.out = d_out8; a.out_plane = (size_t)cout * hw; a.out_f32 = d_out_tc; a.slope = slope;
    a.H = h; a.W = w; a.Cin = cin; a.Cout = cout; a.N = N; a.split_in = split; a.split_out = split;
    a.epi = (mode == 0 || mode == 4) ? TC_EPI_C8 : TC_EPI_DECONV;
    a.k5 = mode == 4;
    a.res_mode = res ? 1 : 0;
    a.act_mode = (mode == 0 || mode == 4) ? 1 : 0;
    a.ocs = ocs; a.ps = ps;
    a.out_planes = planes5 ? 5 : 0;
    int r = launch_tc_conv(a, d_in8, st);
    if (r) { fprintf(stderr, "launch_tc_conv failed: %d\n", r); return RIFE_B200_ERR_INTERNAL; }
    if (mode == 0 || mode == 4) launch_c8_to_planar(d_out8, d_out_tc, cout, h, w, split, st);
    // fp32 CUDA-core reference
    {
        int ocpad = (cout + 63) / 64 * 64;
        std::vector<float> t;
        ConvArgs c;
        memset(&c, 0, sizeof c);
        if (mode == 0 || mode == 4) {
            t.assign((size_t)cin * kk * ocpad, 0.f);
            for (int oc = 0; oc < cout; oc++) for (int ic = 0; ic < cin; ic++) for (int k = 0; k < kk; k++) t[((size_t)ic * kk + k) * ocpad + oc] = wq[((size_t)oc * cin + ic) * kk + k];
        } else {
            t.assign((size_t)4 * cin * 4 * ocpad, 0.f);
            for (int p = 0; p < 4; p++) for (int ic = 0; ic < cin; ic++) for (int rr = 0; rr < 2; rr++) for (int cc = 0; cc < 2; cc++) {
                int ky = 3 - (p >> 1) - 2 * rr, kx = 3 - (p & 1) - 2 * cc;
                for (int oc = 0; oc < cout; oc++) t[(((size_t)p * cin + ic) * 4 + rr * 2 + cc) * ocpad + oc] = wq[((size_t)oc * cin + ic) * 16 + ky * 4 + kx];
            }
        }
        cudaMalloc(&d_wT, t.size() * 4);
        cudaMemcpy(d_wT, t.data(), t.size() * 4, cudaMemcpyHostToDevice);
        c.in = d_in; c.wT = d_wT; c.bias = d_bias; c.Cin = cin; c.H = h; c.W = w; c.Cout = cout; c.ocpad = ocpad;
        if (mode == 0 || mode == 4) {
            c.out = d_out_ref; c.OH = h; c.OW = w; c.DH = h; c.DW = w; c.in_off_y = c.in_off_x = mode == 4 ? -2 : -1; c.out_mul = 1; c.nparity = 1;
            c.res = self_res ? d_in : d_res; c.post_act = 2; c.post_p0 = slope;
            launch_conv(c, mode == 4 ? 5 : 3, 1, st);
        } else {
            c.out = d_tmp; c.OH = 2 * h; c.OW = 2 * w; c.DH = h; c.DW = w; c.in_off_y = c.in_off_x = -1; c.out_mul = 2; c.nparity = 4;
            launch_conv(c, 2, 1, st);
            if (ps > 1) launch_pixelshuffle(d_tmp, cout, 2 * h, 2 * w, d_out_ref, ps, st);
            else cudaMemcpyAsync(d_out_ref, d_tmp, out_elems * 4, cudaMemcpyDeviceToDevice, st);
        }
    }
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { fprintf(stderr, "selftest_conv: %s\n", cudaGetErrorString(e)); return RIFE_B200_ERR_DEVICE; }
    cudaMemcpy(out_tc, d_out_tc, out_elems * 4, cudaMemcpyDeviceToHost);
    cudaMemcpy(out_ref, d_out_ref, out_elems * 4, cudaMemcpyDeviceToHost);
    cudaFree(d_in); cudaFree(d_res); cudaFree(d_bias); cudaFree(d_biasN); cudaFree(d_out_tc); cudaFree(d_out_ref); cudaFree(d_wT); cudaFree(d_tmp);
    cudaFree(d_in8); cudaFree(d_res8); cudaFree(d_out8); cudaFree(d_wpk);
    return RIFE_B200_OK;
    GUARD_END
}

// diagnostics (host only, no GPU needed): parse one network of a model directory
extern "C" int rife_b200_debug_parse_model(const char* param_path, const char* bin_path, int* layers, int* blobs, unsigned long long* weight_values,
                                           char* err, int err_len) {
    GUARD_BEGIN
    if (!param_path || !bin_path) return RIFE_B200_ERR_ARG;
    rife::Net net;
    std::string e;
    int r = rife::load_net(param_path, bin_path, net, e);
    if (err && err_len > 0) { snprintf(err, (size_t)err_len, "%s", e.c_str()); }
    if (r) return RIFE_B200_ERR_MODEL;
    unsigned long long nv = 0;
    for (const rife::Layer& L : net.layers) nv += L.weight.size() + L.bias.size() + L.slope.size();
    if (layers) *layers = (int)net.layers.size();
    if (blobs) *blobs = (int)net.blob_names.size();
    if (weight_values) *weight_values = nv;
    return 0;
    GUARD_END
}

// diagnostics (host only, no GPU needed): the tensor-core weight packing, so a CPU test can replay the MMA operand views
extern "C" int rife_b200_debug_pack_weights(int mode, int cout, int cin, int N, int ocs, int paired, const float* w, unsigned short* out, size_t out_elems) {
    GUARD_BEGIN
    using namespace rife;
    if (!w || !out || cin % 16 || N % 16 || cout <= 0 || cout > N || paired < -1 || paired > 1) return RIFE_B200_ERR_ARG;
    std::vector<uint16_t> pk;
    if (mode == 0) pack_conv3x3_weights(w, cout, cin, N, pk, paired);
    else if (mode == 1) { if (4 * ocs > N || cout > ocs) return RIFE_B200_ERR_ARG; pack_deconv4x4_weights(w, cout, cin, ocs, N, pk, paired); }
    else return RIFE_B200_ERR_ARG;
    if (pk.size() != out_elems) return RIFE_B200_ERR_ARG;
    memcpy(out, pk.data(), pk.size() * sizeof(uint16_t));
    return 0;
    GUARD_END
}

extern "C" int rife_b200_bench_conv(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int iters);
extern "C" int rife_b200_bench_conv_batched(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int batch, int iters);

extern "C" int rife_b200_set_stream(rife_b200_t* h, void* cuda_stream) {
    GUARD_BEGIN
    if (!h) return RIFE_B200_ERR_ARG;
    h->eng->set_stream((cudaStream_t)cuda_stream);
    return RIFE_B200_OK;
    GUARD_END
}

static unsigned long long* g_dbg_dev = nullptr;
static int g_dbg_skip = 0;

// diagnostics: per-CTA clock64 timeline of one tcgen05 conv launch (64 slots per CTA, see tc_conv.cu)
extern "C" int rife_b200_debug_conv_timeline(int gpuid, int cin, int cout, int h, int w, int split, unsigned long long* host_out, int max_ctas) {
    GUARD_BEGIN
    if (!host_out || max_ctas <= 0 || (split >> 24) != 0) return RIFE_B200_ERR_ARG;
    if (cudaSetDevice(gpuid) != cudaSuccess) return RIFE_B200_ERR_DEVICE;
    size_t bytes = (size_t)max_ctas * 64 * 8;
    cudaMalloc(&g_dbg_dev, bytes);
    cudaMemset(g_dbg_dev, 0, bytes);
    // split: bit 0 = split operands, bits 8-15 = images per launch (0 -> 1), bits 16-23 = tiles to skip before recording, bits 24-31 = 0
    const int batch = ((split >> 8) & 0xff) ? ((split >> 8) & 0xff) : 1;
    g_dbg_skip = (split >> 16) & 0xff;
    int r = rife_b200_bench_conv_batched(gpuid, nullptr, cin, cout, h, w, split & 1, batch, 3);  // warm (dbg active on every launch; last one kept)
    cudaDeviceSynchronize();
    cudaMemcpy(host_out, g_dbg_dev, bytes, cudaMemcpyDeviceToHost);
    cudaFree(g_dbg_dev);
    g_dbg_dev = nullptr;
    g_dbg_skip = 0;
    return r;
    GUARD_END
}

extern "C" int rife_b200_bench_conv(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int iters) {
    return rife_b200_bench_conv_batched(gpuid, cuda_stream, cin, cout, h, w, split, 1, iters);
}

extern "C" int rife_b200_bench_conv_batched(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int batch, int iters) {
    GUARD_BEGIN
    using namespace rife;
    if (cin % 16 || cout % 16 || cin <= 0 || h <= 0 || w <= 0 || iters <= 0 || batch < 1 || batch > 16) return RIFE_B200_ERR_ARG;
    h *= batch;  // the synthetic tensors below are allocated as one tall image and then addressed as `batch` images
    if (cudaSetDevice(gpuid) != cudaSuccess) return RIFE_B200_ERR_DEVICE;
    struct Cache { int cin = 0, cout = 0, h = 0, w = 0, split = -1; __half *in8 = 0, *out8 = 0, *wpk = 0; float* bias = 0; };
    static Cache c;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t hw = (size_t)h * w;
    if (c.cin != cin || c.cout != cout || c.h != h || c.w != w || c.split != split) {
        cudaFree(c.in8); cudaFree(c.out8); cudaFree(c.wpk); cudaFree(c.bias);
        std::vector<float> wq((size_t)cout * cin * 9);
        uint32_t s = 12345u;
        for (auto& v : wq) { s = s * 1664525u + 1013904223u; v = __half2float(__float2half_rn(((s >> 9) & 1023) / 1024.f * 0.02f - 0.01f)); }
        std::vector<uint16_t> pk;
        pack_conv3x3_weights(wq.data(), cout, cin, cout, pk);
        std::vector<float> x((size_t)cin * hw), b(cout, 0.01f);
        for (auto& v : x) { s = s * 1664525u + 1013904223u; v = ((s >> 9) & 1023) / 1024.f - 0.5f; }
        float* d_x = 0;
        cudaMalloc(&d_x, x.size() * 4); cudaMalloc(&c.in8, x.size() * 4); cudaMalloc(&c.out8, (size_t)cout * hw * 4);
        cudaMalloc(&c.wpk, pk.size() * 2); cudaMalloc(&c.bias, cout * 4);
        cudaMemcpy(d_x, x.data(), x.size() * 4, cudaMemcpyHostToDevice);
        cudaMemcpy(c.wpk, pk.data(), pk.size() * 2, cudaMemcpyHostToDevice);
        cudaMemcpy(c.bias, b.data(), cout * 4, cudaMemcpyHostToDevice);
        launch_planar_to_c8(d_x, c.in8, cin, h, w, split, 0);
        cudaDeviceSynchronize();
        cudaFree(d_x);
        c.cin = cin; c.cout = cout; c.h = h; c.w = w; c.split = split;
    }
    TcConvArgs a;
    memset(&a, 0, sizeof a);
    a.wpk = c.wpk; a.bias = c.bias; a.out = c.out8; a.out_plane = (size_t)cout * hw; a.slope = 0.2f;
    a.res = cin == cout ? c.in8 : nullptr; a.res_plane = (size_t)cin * hw; a.res_split = split; a.res_mode = cin == cout ? 1 : 0;
    a.H = h; a.W = w; a.Cin = cin; a.Cout = cout; a.N = cout; a.split_in = split; a.split_out = split; a.epi = TC_EPI_C8; a.act_mode = 1;
    a.dbg = g_dbg_dev;
    a.dbg_skip = g_dbg_skip;
    if (batch > 1) {
        // reinterpret the tall synthetic tensor as `batch` images: per image [planes][C/8][h/batch][w][8]; the values are
        // arbitrary, only the addressing pattern matters for timing
        a.H = h / batch;
        a.batch = batch;
        a.in_bstride = a.res_bstride = a.out_bstride = (size_t)cin * (h / batch) * w * 2;
        a.out_plane = a.res_plane = (size_t)cout * (h / batch) * w;
    }
    for (int i = 0; i < iters; i++) {
        int r = launch_tc_conv(a, c.in8, st);
        if (r) return RIFE_B200_ERR_INTERNAL;
    }
    return cudaGetLastError() == cudaSuccess ? RIFE_B200_OK : RIFE_B200_ERR_DEVICE;
    GUARD_END
}

// ---- diagnostics of the HBM-side kernels (hbm_kernels.cu) ---------------------------------------------------------------
// which: 0 preproc (c = orientations 1 | 8; in = u8 [h][w][3]; out = float [c][3][hp][wp], orientations >= 4 transposed)
//        1 postproc (c = inputs 1 | 2 | 8 | 16; in = float [c][3][hp*wp], input i in orientation i & 7; out = u8 [h][w][3])
//        2 flow_tta_avg (c = channels 2 | 4 | 5; in = 8 blobs of c planes of h x w (blobs 4-7 transposed); out = same, averaged)
//        3 warp (in = float [c][h][w], in2 = flow [2][h][w]; out = float [c][h][w])
//        4 temporal_merge_v2 (c = has_mask; in = f, in2 = fr, 4 + c planes of w*h; out = f' followed by fr')
//        5 temporal_merge_v1 (2 planes)
// iters > 0: timing mode -- synthetic device-resident data, the kernel is launched `iters` times on `cuda_stream`, nothing is
// copied (in / in2 / out may be NULL).  iters == 0: test mode -- one launch on the host data, result copied back.
extern "C" int rife_b200_debug_hbm(int gpuid, void* cuda_stream, int which, int w, int h, int c, int iters, const void* in, const void* in2, void* out) {
    GUARD_BEGIN
    using namespace rife;
    if (w <= 0 || h <= 0 || c < (which == 4 ? 0 : 1) || which < 0 || which > 5 || iters < 0) return RIFE_B200_ERR_ARG;
    if (iters == 0 && (!in || !out)) return RIFE_B200_ERR_ARG;
    if (cudaSetDevice(gpuid) != cudaSuccess) return RIFE_B200_ERR_DEVICE;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int wp = (w + 31) / 32 * 32, hp = (h + 31) / 32 * 32;
    const size_t plane = (size_t)wp * hp, n = (size_t)w * h;
    size_t in_b = 0, in2_b = 0, out_b = 0;
    switch (which) {
        case 0: in_b = n * 3; out_b = (size_t)c * 3 * plane * 4; break;
        case 1: in_b = (size_t)c * 3 * plane * 4; out_b = n * 3; break;
        case 2: in_b = out_b = (size_t)8 * c * n * 4; break;
        case 3: in_b = out_b = (size_t)c * n * 4; in2_b = 2 * n * 4; break;
        case 4: in_b = in2_b = (size_t)(4 + (c ? 1 : 0)) * n * 4; out_b = 2 * in_b; break;
        default: in_b = in2_b = 2 * n * 4; out_b = 2 * in_b; break;
    }
    // timing mode keeps its buffers between calls of the same shape (bench loops); test mode allocates and frees
    struct Cache { int which = -1, w = 0, h = 0, c = 0; void *a = 0, *b = 0, *o = 0; };
    static Cache cache;
    void *d_in = 0, *d_in2 = 0, *d_out = 0;
    const bool timing = iters > 0;
    bool fresh = true;  // in-place kernels (2, 4, 5): the working copy is initialised once per buffer set, never inside a timed call
    if (timing && cache.which == which && cache.w == w && cache.h == h && cache.c == c) { d_in = cache.a; d_in2 = cache.b; d_out = cache.o; fresh = false; }
    else {
        if (timing) { cudaFree(cache.a); cudaFree(cache.b); cudaFree(cache.o); cache = Cache(); }
        if (cudaMalloc(&d_in, in_b) != cudaSuccess || (in2_b && cudaMalloc(&d_in2, in2_b) != cudaSuccess) || cudaMalloc(&d_out, out_b) != cudaSuccess) {
            cudaFree(d_in); cudaFree(d_in2); cudaFree(d_out);
            return RIFE_B200_ERR_DEVICE;
        }
        if (timing) {
            cudaMemset(d_in, which == 0 ? 0x5a : 0, in_b);  // flows of zero: the warp gathers its own pixel (best-case locality is what a smooth flow gives)
            if (d_in2) cudaMemset(d_in2, 0, in2_b);
            cache.which = which; cache.w = w; cache.h = h; cache.c = c; cache.a = d_in; cache.b = d_in2; cache.o = d_out;
        } else {
            cudaMemcpy(d_in, in, in_b, cudaMemcpyHostToDevice);
            if (d_in2) cudaMemcpy(d_in2, in2, in2_b, cudaMemcpyHostToDevice);
        }
    }
    const int reps = timing ? iters : 1;
    for (int it = 0; it < reps; it++) {
        switch (which) {
            case 0: launch_preproc((const uint8_t*)d_in, w, h, (float*)d_out, wp, hp, c, 0, st); break;
            case 1: {
                const float* ins[16];
                for (int i = 0; i < c && i < 16; i++) ins[i] = (const float*)d_in + (size_t)i * 3 * plane;
                launch_postproc(ins, c, wp, hp, (uint8_t*)d_out, w, h, 0, 0, st);
                break;
            }
            case 2: {
                float* f8[8];
                if (fresh && it == 0) cudaMemcpyAsync(d_out, d_in, in_b, cudaMemcpyDeviceToDevice, st);
                for (int i = 0; i < 8; i++) f8[i] = (float*)d_out + (size_t)i * c * n;
                launch_flow_tta_avg(f8, c, w, h, st);
                break;
            }
            case 3: launch_warp((const float*)d_in, (const float*)d_in2, (float*)d_out, c, h, w, st); break;
            case 4:
            case 5: {
                if (fresh && it == 0) {
                    cudaMemcpyAsync(d_out, d_in, in_b, cudaMemcpyDeviceToDevice, st);
                    cudaMemcpyAsync((char*)d_out + in_b, d_in2, in_b, cudaMemcpyDeviceToDevice, st);
                }
                if (which == 4) launch_temporal_merge_v2((float*)d_out, (float*)((char*)d_out + in_b), n, c ? 1 : 0, st);
                else launch_temporal_merge_v1((float*)d_out, (float*)((char*)d_out + in_b), n, st);
                break;
            }
        }
    }
    if (timing) return cudaGetLastError() == cudaSuccess ? RIFE_B200_OK : RIFE_B200_ERR_DEVICE;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaMemcpy(out, d_out, out_b, cudaMemcpyDeviceToHost);
    cudaFree(d_in); cudaFree(d_in2); cudaFree(d_out);
    return e == cudaSuccess ? RIFE_B200_OK : RIFE_B200_ERR_DEVICE;
    GUARD_END
}
