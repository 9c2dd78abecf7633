// fused_v46.h -- hand-scheduled fast path for the 4-block IFNet of the rife-v4 family (rife-v4.6 and rife-v4; see fused_v46.cu)
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "exec.h"
#include "model.h"

namespace rife {

constexpr int V46_MAX_BATCH = 8;
struct StageTimer;

class V46Runner {
public:
    ~V46Runner();
    // `weights` = the NetRunner that owns the packed tensor-core weights of `net` on this device
    int init(const Net* net, const NetRunner* weights, std::string& err);
    bool ok() const { return ok_; }
    // bit k set: the residual chain of IFBlock k runs on plain fp16 activations (half the tensor work, ~2^-11 operand
    // rounding); 0 = every tensor-core activation is split hi+lo
    void set_plain_mask(int m) { plain_mask_ = m & 255; }
    // 0: flow / mask planes stored at full resolution between the block-2 head and the tail; 1: block-3 head stops
    // storing them; 2: never stored, rebuilt from the per-block flow tensors where needed (same arithmetic, fewer HBM bytes)
    void set_recompute(int m) { recompute_ = m < 0 ? 0 : (m > 2 ? 2 : m); }
    // 1: reproduce the reference CPU path's contiguous read of the padded output (src/rife.cpp:4375-4387) instead of cropping
    void set_crop_quirk(int q) { crop_quirk_ = q != 0; }
    // 1: block-head tensors in the packed form (one fp16 plane; only the flow channels keep a lo part): fused_v46_kernels.cuh
    void set_head_pack(int p) { head_pack_ = p != 0; }
    void set_bgr(int b) { bgr_ = b != 0; }  // frames are B,G,R in memory (the reference's Windows build)
    bool is_v4() const { return v4_; }
    // per-stage CUDA-event times of run_batch (diagnostics / bench.py's breakdown; synchronises the stream after every batch)
    void set_ktime(int on);
    std::string stage_report() const;
    int run(const uint8_t* d_in0, const uint8_t* d_in1, int w, int h, float t, uint8_t* d_out, cudaStream_t st, std::string& err);
    int run_batch(int n, const uint8_t* const* d_in0, const uint8_t* const* d_in1, int w, int h, const float* ts, uint8_t* const* d_out, cudaStream_t st,
                  std::string& err);

private:
    int ensure(int w, int h, int batch, std::string& err);
    int conv(int slot, const __half* in, __half* out, const __half* res, float* out_f32, int oh, int ow, bool out_s2d, int batch, bool split_in,
             bool split_out, cudaStream_t st);
    // activation / residual form of each of the 44 convolutions, read from the graph at init()
    struct ConvCfg {
        int layer = -1;
        int act_mode = 0;            // 0 none, 1 leaky(slope), 2 per-channel PReLU
        float slope = 0.f;
        const float* prelu = nullptr;
        int res_mode = 0;            // residual chain: 1 = add before the activation (v4.6, every conv), 2 = add after it (v4, last conv)
    };
    ConvCfg cfg_[44];
    bool v4_ = false;                // rife-v4 layout: 5-channel flow heads at half the block resolution, PReLU, one residual per chain
    int crop_quirk_ = 0, bgr_ = 0, head_pack_ = 0;
    __half* wpk_head_[4] = {};
    StageTimer* tm_ = nullptr;
    const Net* net_ = nullptr;
    const NetRunner* wr_ = nullptr;
    bool ok_ = false;
    int plain_mask_ = 0;
    int recompute_ = 0;
    std::vector<int> conv_;  // the 44 conv / deconv layer indices in graph order
    int wp_ = 0, hp_ = 0, cap_ = 0;
    std::vector<void*> bufs_;
    uchar4* rgbx_ = nullptr;  // the distinct frames of a batch, padded RGBX
    float *F_ = nullptr, *M_ = nullptr, *d_[4] = {};
    __half *x_[4] = {}, *y0_[4] = {}, *a_[4] = {}, *b_[4] = {}, *c_[4] = {};
    bool res_split_ = false;  // the residual handed to conv() carries a lo plane
};

}  // namespace rife
