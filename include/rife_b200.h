/* rife_b200.h -- C ABI of librife_b200.so, the B200-native replacement for the engine underneath the
 * reference's `class RIFE` (/root/reference/src/rife.h:11-52).  Plain pointers and sizes only; every entry
 * point returns 0 on success and a negative code on error, never throws, and is safe to call from several
 * threads on the same handle (the reference calls RIFE::process concurrently from its `proc` threads,
 * /root/reference/src/main.cpp:346-366).
 *
 * What each entry point replaces:
 *   rife_b200_device_count   ncnn::get_gpu_count()                       src/main.cpp:782-799
 *   rife_b200_create         RIFE::RIFE(gpuid, tta, tta_temporal, uhd,   src/rife.cpp:27-47, call site main.cpp:825
 *                                       num_threads, rife_v2, rife_v4)
 *   rife_b200_load           RIFE::load(modeldir)                        src/rife.cpp:127-379, call site main.cpp:827
 *   rife_b200_load_w         RIFE::load(const std::wstring&)             src/rife.cpp:80-110 (the Windows build's overload)
 *   rife_b200_process        RIFE::process(in0, in1, timestep, out)      src/rife.cpp:381-405, call site main.cpp:360
 *   rife_b200_destroy        RIFE::~RIFE()                               src/rife.cpp:49-78
 * Additions for the stream / benchmark path (no reference counterpart; the reference re-uploads per call):
 *   rife_b200_process_device     same computation with frames already resident in device memory
 *   rife_b200_process_batch      n independent pairs, pipelined over the handle's streams
 *   rife_b200_weights_* / rife_b200_load_packed   rank-0 parses + packs the model, the blob is broadcast
 *                                (NCCL over NVLink by the caller, one process per GPU) and loaded without
 *                                touching the model directory (SURVEY.md section 8e)
 *
 * gpuid == -1 (the reference's CPU mode) is rejected: there is no CPU fallback in this library.
 */
#ifndef RIFE_B200_H
#define RIFE_B200_H

#include <stddef.h>
#include <wchar.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rife_b200 rife_b200_t;

#define RIFE_B200_OK 0
#define RIFE_B200_ERR_ARG (-1)      /* bad argument (null pointer, w/h <= 0, gpuid < 0, ...) */
#define RIFE_B200_ERR_DEVICE (-2)   /* no such CUDA device / CUDA runtime failure */
#define RIFE_B200_ERR_MODEL (-3)    /* model directory unreadable or malformed */
#define RIFE_B200_ERR_STATE (-4)    /* process before load */
#define RIFE_B200_ERR_INTERNAL (-5)

int rife_b200_device_count(void);

int rife_b200_create(rife_b200_t** handle, int gpuid, int tta_mode, int tta_temporal_mode, int uhd_mode,
                     int num_threads /* ignored: kept for signature parity */, int rife_v2, int rife_v4);

/* reads flownet.{param,bin} (+ contextnet / fusionnet unless rife_v4), as the reference does */
int rife_b200_load(rife_b200_t* handle, const char* modeldir);
/* wide-character path (the reference's Windows overload); converted to UTF-8 */
int rife_b200_load_w(rife_b200_t* handle, const wchar_t* modeldir);

/* in0/in1/out: packed RGB u8, HWC, w*h*3 bytes each, caller-owned HOST memory.
 * timestep == 0 / 1 copies in0 / in1 to out (the reference rebinds the output Mat, src/rife.cpp:3206-3216). */
int rife_b200_process(rife_b200_t* handle, const unsigned char* in0_rgb, const unsigned char* in1_rgb,
                      int w, int h, float timestep, unsigned char* out_rgb);

/* same, with all three buffers in DEVICE memory of the handle's GPU; asynchronous work is complete on return */
int rife_b200_process_device(rife_b200_t* handle, const unsigned char* d_in0_rgb, const unsigned char* d_in1_rgb,
                             int w, int h, float timestep, unsigned char* d_out_rgb);

/* n independent frame pairs (host memory), same w/h; pairs are pipelined (H2D / compute / D2H overlap) */
int rife_b200_process_batch(rife_b200_t* handle, int n, const unsigned char* const* in0_rgb,
                            const unsigned char* const* in1_rgb, int w, int h, const float* timesteps,
                            unsigned char* const* out_rgb);

/* n independent pairs with all buffers in DEVICE memory; pairs are dealt to the handle's concurrent lanes
 * (option "lanes", default 2) so small layers of different pairs overlap on the GPU */
int rife_b200_process_batch_device(rife_b200_t* handle, int n, const unsigned char* const* d_in0_rgb,
                                   const unsigned char* const* d_in1_rgb, int w, int h, const float* timesteps,
                                   unsigned char* const* d_out_rgb);

/* precision tier: 0 = exact (fp32 CUDA-core path for every layer), 1 = fast (tcgen05 fp16 tensor-core
 * convolutions with split-precision operands where needed).  Default 1 when the model supports it. */
/* other keys: "lanes" (1-8 concurrent streams; default 2, 8 for spatial-TTA engines, whose 8 orientations are dealt to the lanes), "batch" (pairs per lock-step batch on the fused path, 0 = auto),
 * "plain_blocks" (bit k: IFBlock k's residual chain uses plain fp16 activations instead of split hi+lo; default 12),
 * "fast" (0/1 fused rife-v4.6 path), "async" (0/1), "fuse" (0/1 epilogue fusion in the fp32 path),
 * "combine" (0/1, default 1: concurrent rife_b200_process calls on one handle run as one lock-step batch),
 * "recompute_fm" (0-2, default 0: fused path rebuilds the full-resolution flow / mask planes instead of storing them),
 * "cpu_crop_quirk" (0/1, default 0).  The output frame is the w x h crop of the padded result, as the reference's GPU path
 *   produces it (src/rife_postproc.comp:42).  The reference's CPU path instead reads the first w*h floats of every padded
 *   channel contiguously (src/rife.cpp:4375-4387), which shears the frame whenever w % 32 != 0; 1 reproduces that
 *   byte for byte (used by the parity tests against the reference's -g -1 binary).  No difference when w % 32 == 0.
 * "bgr" (0/1, default 0): frame bytes are B,G,R -- the reference's Windows build (src/rife_preproc.comp:13,53-56),
 * "frame_cache" (0/1, default 0): input frames uploaded by rife_b200_process / _process_batch stay on the device and are
 *   found again by host pointer in later calls (pair (k, k+1) then uploads only frame k+1).  The caller must not modify
 *   or free-and-reuse a frame buffer it has handed in until rife_b200_forget_frames() or "frame_cache" = 0.
 *   Within one call a frame shared by several pairs is always uploaded once.
 * "stage_pageable" (0/1, default 1): rife_b200_process calls that arrive with pageable buffers (what the reference CLI passes)
 *   copy their frames through a pinned slot in the CALLING thread, so concurrent callers copy in parallel and the combined
 *   batch runs on asynchronous DMA only; ignored while "frame_cache" is on. */
int rife_b200_set_option(rife_b200_t* handle, const char* key, int value);
/* reads back "precision", "lanes", "fast" (requested) and "fast_active" (1 when the fused rife-v4.6 path passed its
 * load-time self-check against the generic executor and is the one process() runs) */
int rife_b200_get_option(rife_b200_t* handle, const char* key, int* value);

/* Diagnostics: with option "ktime" = 1 the fused path records CUDA-event times of every stage of a lock-step batch (the
 * stream is synchronised after each batch while it is on).  Text, one block per lane: "lane\t<i>", "batches\t<n>", then
 * "<stage>\t<microseconds per batch>\t<kernel launches per batch>" per stage.  bench.py's per-stage breakdown. */
int rife_b200_stage_report(rife_b200_t* handle, char* buf, size_t cap);

/* drops every cached input frame (option "frame_cache") */
int rife_b200_forget_frames(rife_b200_t* handle);

/* packed-weights path for multi-GPU loading without re-reading the model directory on every rank */
int rife_b200_weights_size(rife_b200_t* handle, size_t* bytes);                 /* after load() on rank 0 */
int rife_b200_weights_export(rife_b200_t* handle, void* host_dst, size_t bytes);
int rife_b200_load_packed(rife_b200_t* handle, const void* host_src, size_t bytes);

/* Run the handle's work on a caller-owned CUDA stream (cudaStream_t passed as void*; NULL restores the handle's own
 * stream) so a caller can bracket it with its own events.  option "async" = 1 makes rife_b200_process_device return
 * without synchronising that stream. */
int rife_b200_set_stream(rife_b200_t* handle, void* cuda_stream);

/* Launches the tcgen05 conv3x3 (cin -> cout, h x w, bias + residual + leaky) `iters` times on `cuda_stream` with
 * device-resident synthetic data and returns; used by bench.py to time the dominant kernel with its own events. */
int rife_b200_bench_conv(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int iters);
/* same with `batch` images per launch (the lock-step batch of the fused path) */
int rife_b200_bench_conv_batched(int gpuid, void* cuda_stream, int cin, int cout, int h, int w, int split, int batch, int iters);

/* Diagnostics: clock64 timeline (64 slots per CTA) of one tcgen05 conv launch; see csrc/tc_conv.cu for the slot map.
 * `split`: bit 0 = split hi+lo operands, bits 8-15 = images per launch (0 = 1), bits 16-23 = tiles each CTA skips
 * before recording (steady state instead of pipeline fill); the bits above must be 0 (RIFE_B200_ERR_ARG otherwise). */
int rife_b200_debug_conv_timeline(int gpuid, int cin, int cout, int h, int w, int split, unsigned long long* host_out,
                                  int max_ctas);

/* Diagnostics: runs ONE convolution layer through the tcgen05 tensor-core kernel and through the fp32 CUDA-core
 * kernel on the same data and returns both results (planar fp32, host memory) so a test can compare them.
 * mode 0: conv3x3 s1 p1 (+bias, + optional residual `res`, + leaky `slope`), in [cin][h][w] -> out [cout][h][w];
 *         res == in (same pointer, cin == cout) exercises the self-residual path (identity tap on the tensor core)
 * mode 1: deconv4x4 s2 p1 (+bias) followed by PixelShuffle(ps), in [cin][h][w] -> out [cout/(ps*ps)][2h*ps][2w*ps]
 * mode 3: mode 1 with cout = 24, ps = 2, storing only the first five output planes (the IFNet flow head; plane 5 of
 *         out_tc is left untouched)
 * mode 4: conv5x5 s1 p2 (+bias, + optional residual, + leaky), weight [cout][cin][5][5] (the 5x5 row-stage variant of the kernel)
 * split != 0 stores activations as split-fp16 (hi+lo) for the tensor-core path. */
int rife_b200_selftest_conv(int gpuid, int mode, int cin, int cout, int h, int w, int split, int ps, const float* in,
                            const float* weight, const float* bias, const float* res, float slope, float* out_tc,
                            float* out_ref);

/* Diagnostics: the HBM-side kernels of the generic path (csrc/hbm_kernels.cu) on caller data (iters == 0: one launch, result
 * copied back; used by tests/test_hbm_kernels_gpu.py against numpy restatements) or on device-resident synthetic data
 * (iters > 0: `iters` launches on `cuda_stream`, nothing copied; used by tools/bench_hbm.py for GB/s and ncu captures).
 * which: 0 preproc (c = orientations), 1 postproc (c = inputs), 2 flow_tta_avg (c = channels), 3 warp (c = channels),
 * 4 temporal_merge_v2 (c = has_mask), 5 temporal_merge_v1; buffer layouts: see csrc/capi.cu. */
int rife_b200_debug_hbm(int gpuid, void* cuda_stream, int which, int w, int h, int c, int iters, const void* in, const void* in2,
                        void* out);

/* Diagnostics (host only, no GPU): parses one network (<name>.param + <name>.bin, the reference's model format:
 * src/ncnn/src/net.cpp:1374-1590, modelbin.cpp:89-260) and reports its layer / blob / weight-value counts; on failure
 * returns RIFE_B200_ERR_MODEL with the loader's message in `err` (may be NULL). */
int rife_b200_debug_parse_model(const char* param_path, const char* bin_path, int* layers, int* blobs,
                                unsigned long long* weight_values, char* err, int err_len);

/* Diagnostics (host only, no GPU): the weight packing of the tcgen05 kernel, fp16 bit patterns.
 * mode 0: conv3x3 w[cout][cin][3][3]; mode 1: deconv4x4 s2 w[cout][cin][4][4] with `ocs` column slots per output parity.
 * out_elems must be (cin/16)*9*2*N*8.  paired: 0 = [kc][tap][half][N][8]; 1 = [kc][dx][half][3N: dy2|dy0|dy1][8]
 * (the layout of the paired MMA issue; with 2N > 256 the layout of 0); -1 = what the kernel uses for this N (1 when
 * 2N <= 256, else 0).  Any other value returns RIFE_B200_ERR_ARG. */
int rife_b200_debug_pack_weights(int mode, int cout, int cin, int N, int ocs, int paired, const float* w,
                                 unsigned short* out, size_t out_elems);

/* kernels launched by this library since process start (bench.py reports it as gpu_launches) */
unsigned long long rife_b200_launch_count(void);

/* bytes this library copied host->device / device->host since process start (bench.py reports them per step) */
unsigned long long rife_b200_h2d_bytes(void);
unsigned long long rife_b200_d2h_bytes(void);

/* last error message of the handle, copied into a buffer owned by the calling thread (valid until that thread's next call
 * of this function); never NULL */
const char* rife_b200_last_error(rife_b200_t* handle);

void rife_b200_destroy(rife_b200_t* handle);

#ifdef __cplusplus
}
#endif
#endif /* RIFE_B200_H */
