// tc_conv.h -- host interface of the tcgen05 implicit-GEMM convolution (tc_conv.cu)
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace rife {

enum { TC_EPI_C8 = 0, TC_EPI_DECONV = 1 };

struct TcConvArgs {
    const __half* wpk;      // packed weights [Cin/16][9][2][N][8]
    const float* bias;      // [N] (zero padded)
    const __half* res;      // residual in C8 layout (Cout channels) or null
    size_t res_plane;       // element offset of the residual's lo plane
    __half* out;            // C8 output (TC_EPI_C8)
    size_t out_plane;       // element offset of the output's lo plane
    float* out_f32;         // planar fp32 output (TC_EPI_DECONV)
    const float* prelu;     // per-channel slopes (act_mode 2)
    float slope;            // leaky slope (act_mode 1)
    int H, W, Cin, Cout, N; // N = GEMM columns (Cout for conv, 4*ocs for deconv)
    int split_in, split_out, res_split;
    int epi;                // TC_EPI_*
    int res_mode;           // 0 none, 1 add before activation, 2 add after activation (3 is internal: the launcher turns 1 into 3 when res == in)
    int act_mode;           // 0 none, 1 leaky(slope), 2 prelu, 3 sigmoid (deconv epilogue only)
    int ocs, ps;            // deconv: output-channel slots per parity, PixelShuffle factor (1 = none)
    int out_planes;         // deconv + PixelShuffle: store only the first out_planes planes (0 = all)
    int batch;              // images per launch (0 / 1 = single); image b lives at base + b * *_bstride
    size_t in_bstride, res_bstride, out_bstride, outf_bstride;  // elements of the respective tensors
    int k5;                 // 5x5 stride-1 pad-2 convolution (weights from pack_conv5x5_weights)
    int s2;                 // stride-2 conv: `in` is the space-to-depth tensor (4 sub-images of H x W, Cin channels each)
    int out_s2d;            // write the C8 output in space-to-depth form (H, W even)
    int out_cgroups;        // 8-channel groups of the output TENSOR (0 = Cout / 8); larger when this launch writes a channel slice of it
    int tiles_x, tiles_y, num_sms;  // filled by the launcher
    int stages;                     // filled by the launcher: pipeline depth (<= 8)
    int ks;                         // filled by the launcher: 16-channel chunks per pipeline stage (resident-weight kernels)
    int wres;                       // filled by the launcher: the layer's packed weights stay resident in shared memory
    unsigned long long* dbg;        // optional timeline buffer: 64 clock64 slots per CTA (diagnostics)
    int dbg_skip;                   // tiles (per CTA) to skip before the timeline starts recording
};

// `in`: C8 planar activation [planes][Cin/8][H][W][8] fp16.  Returns 0 on success.
int launch_tc_conv(TcConvArgs a, const void* in, cudaStream_t st);
int tc_conv_tile_rows(int N);
// Paired MMA issue over [dy2 | dy0 | dy1] weight blocks for every stride-1 layer whose 2N columns fit one MMA: the weight
// packers and the launcher both decide the layout here.
__host__ __device__ constexpr bool tc_paired(int N) { return 2 * N <= 256; }
constexpr int TC_KS_DEFAULT = 2;  // measured (profiles/r2_s6): chain of IFBlock 3 704 -> 692 us, IFBlock 2 414 -> 403 us per 8 launches

void launch_planar_to_c8(const float* in, __half* out, int C, int H, int W, int split, cudaStream_t st, int Cpad = 0, int s2d = 0);
void launch_c8_to_planar(const __half* in, float* out, int C, int H, int W, int split, cudaStream_t st, int Cpad = 0, int s2d = 0);

// paired: -1 = what the launcher will assume for this N (tc_paired), 0 plain / 1 paired (if 2N <= 256) = explicit (diagnostics)
void pack_conv3x3_weights(const float* w, int cout, int cin, int N, std::vector<uint16_t>& out, int paired = -1);
void pack_conv5x5_weights(const float* w, int cout, int cin, int N, std::vector<uint16_t>& out);
void pack_conv3x3s2_weights(const float* w, int cout, int cin, int cinp, int N, std::vector<uint16_t>& out);
void pack_deconv4x4_weights(const float* w, int cout, int cin, int ocs, int N, std::vector<uint16_t>& out, int paired = -1);

}  // namespace rife
