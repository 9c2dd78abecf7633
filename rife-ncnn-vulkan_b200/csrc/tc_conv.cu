// tc_conv.cu -- 3x3 stride-1 pad-1 convolution (and deconv4x4s2 re-expressed as a 3x3 conv with 4x the output
// channels) as an implicit GEMM on the 5th-gen tensor cores: TMA -> shared memory -> tcgen05.mma (fp16 operands,
// fp32 accumulation in TMEM) -> tcgen05.ld epilogue.  sm_100a only.
//
// Activations live in HBM in the "C8 planar" layout  [plane][C/8][H][W][8] fp16  (plane 0 = hi, plane 1 = lo where
// v ~= hi + lo is the split-fp16 representation of an fp32 value; SURVEY.md Appendix C: split operands reproduce the
// fp32 oracle at its own noise floor, plain fp16 storage does not reach +-1 LSB on every layer).
//
// Work item = a tile of TH x 62 output pixels (TH = 2*MT rows), flattened onto MT accumulators of 128 rows x N
// columns; the A operand of tap (dy,dx) for accumulator m is simply the shared-memory tile viewed from the
// start address  ((2m+dy)*64 + dx) * 16 B  (no-swizzle K-major core matrices: 8 pixels x 16 B contiguous), so one
// halo tile serves all 9 taps.  Out-of-image halo pixels are zero-filled by TMA = the convolution's zero padding.
// Pipeline stage = 16 input channels: A_hi (+A_lo) tile slabs + the weights of all 9 taps for those channels.
//
// Warp roles (192 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2-5 epilogue.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <type_traits>

#include "tc_conv.h"
#include "kernels.h"

namespace rife {

namespace {

constexpr int NTHREADS = 320;  // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quarter)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    // try_wait suspends the thread for a hardware-bounded time; the counter turns a protocol bug (lost arrival,
    // faulted TMA) into a trap after a few seconds instead of a hung GPU
    for (uint32_t spins = 0;; spins++) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
        if (done) return;
        if (spins > (1u << 26)) __trap();
    }
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(smem_u32(dst)),
                 "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
                 "r"(smem_u32(bar))
                 : "memory");
}
// K-major, SWIZZLE_NONE shared-memory matrix descriptor (sm_100 format, version field = 1):
// core matrix = 8 rows x 16 B contiguous; SBO = byte distance between 8-row groups, LBO = between the two 16 B K halves.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Convergent-issue variants: the whole warp executes the asm, elect.sync picks the one lane that issues.  Keeping the
// issuing loop free of thread divergence lets ptxas keep descriptors in uniform registers and emit a bare predicated
// UTCHMMA (a single-lane `if (lane == 0)` loop made it wrap every MMA in an ELECT / BRA.U.ANY lane loop, ~250 cycles each).
__device__ __forceinline__ void umma_f16_elect(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        ".reg .b64 da, db;\n"
        "mov.b64 da, {%1, %2};\n"
        "mov.b64 db, {%3, %4};\n"
        "setp.ne.b32 p, %6, 0;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
        "}\n" ::"r"(tmem_d),
        "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate));
}
#include "tc_mma_issue.inc"

__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n"
        ".reg .pred q;\n"
        "elect.sync _|q, 0xffffffff;\n"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
        "}\n" ::"r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, "
        "%23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// wait::ld variants that name the destination registers as in/out operands: values read after the wait formally depend
// on it, so the compiler cannot schedule a consumer of an in-flight tcgen05.ld above the wait (software-pipelined loads)
__device__ __forceinline__ void tmem_ld_wait_dep16(uint32_t* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                   "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait_dep32(uint32_t* r) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]),
                   "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]),
                   "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]),
                   "+r"(r[31])
                 :
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

struct HalfPack8 {
    uint4 v;
};
__device__ __forceinline__ uint32_t pack2(__half a, __half b) { return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16); }

}  // namespace

// N = UMMA N (output columns per accumulator), MT = accumulators (128 flattened positions each) per tile,
// STAGES = minimum pipeline depth; the launcher raises it (TcConvArgs::stages, up to 8) to what shared memory allows.
// TAPS = 9: stride-1 conv (every K chunk uses the 9 shifted views).  TAPS = 4: stride-2 conv over a space-to-depth
// input (4 parity sub-images [py][px] of H/2 x W/2, each a run of K chunks): input row 2y+dy-1 is row y-1 of the odd
// sub-image for dy = 0, row y of the even one for dy = 1 and row y of the odd one for dy = 2 (columns alike), so a
// chunk of parity (py,px) contributes (py?2:1)*(px?2:1) taps, each again a plain shifted view of the same slab.
template <int N, int MT, int STAGES, int TAPS>
__global__ void __launch_bounds__(NTHREADS, 1) tc_conv3x3_kernel(const __grid_constant__ CUtensorMap tmA, TcConvArgs a) {
    // TAPS = 5: a 5x5 stride-1 pad-2 convolution, one KERNEL ROW per pipeline stage.  The K loop runs over (16-channel chunk,
    // dy): a stage carries the 2*MT image rows that tap row dy reads (no halo rows: the next dy re-loads the rows shifted by
    // one, from L2) and the weights of its five taps, whose A operands are the slab viewed from start column dx = 0..4.
    // The tile keeps 60 valid columns (halo 2 left and right).  All 25 taps of a chunk in one stage would need up to 150 KB of
    // weights per stage (N = 192); a row is 31 KB.
    constexpr int HALO = TAPS == 5 ? 2 : 1;
    constexpr int TWP = 64;                       // tile width incl. the halo columns left and right
    constexpr int TVALID = TWP - 2 * HALO;
    constexpr int ROWS = TAPS == 5 ? 2 * MT : 2 * MT + 2;  // input rows per stage (3x3: halo rows included)
    constexpr int A_PLANE = 2 * ROWS * TWP * 16;  // bytes of one plane slab: 2 eight-channel halves
    constexpr int W_BYTES = TAPS * 2 * N * 16;
    constexpr int ACC_COLS = MT * N;              // TMEM columns per accumulator set
    static_assert(2 * ACC_COLS <= 512, "TMEM overflow");
    static_assert(N % 16 == 0 && N >= 16 && N <= 256, "invalid UMMA N");

    extern __shared__ __align__(1024) uint8_t smem[];
    const int nplanes = a.split_in ? 2 : 1;
    // a.wres: the packed weights of the whole layer stay in shared memory for the life of the (persistent) CTA and a
    // pipeline stage carries activations only; otherwise every stage re-streams its 16-channel weight slice from L2
    // (per tile that is more bytes than the activations themselves).
    // a.ks > 1 (resident weights only): a pipeline stage carries ks consecutive 16-channel chunks (sub-slabs), i.e. one barrier
    // round trip (full / empty) per ks chunks instead of per chunk
    const int sub_bytes = ((A_PLANE * nplanes + (a.wres ? 0 : W_BYTES)) + 1023) & ~1023;
    const int KS = a.ks > 1 ? a.ks : 1;
    const int stage_bytes = sub_bytes * KS;
    const int NST = a.stages;  // pipeline depth (<= 8), chosen by the launcher
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + (size_t)NST * stage_bytes + 1024);  // +1024: overrun pad for the last tap of the last slab
    uint64_t* empty = full + 8;
    uint64_t* acc_full = empty + 8;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* wbar = acc_empty + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(wbar + 1);
    float* slope_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full) + 256);  // per-channel (slope - 1), PReLU epilogue only; 16-byte aligned
    // Constant MMA operands, built once per CTA:
    //  ones  : A tile 128 x 16 with K columns 0..2 = 1      }  first MMA of every tile: D = ones * biasB = the fp32 bias
    //  biasB : B tile 16 x N, K rows 0..2 = bias as hi+lo+lo2 }  (three fp16 pieces), so no epilogue touches the bias
    //  ident : res_mode 3 (residual == this conv's own input): the residual is added by the tensor core as a tenth tap
    //          whose B operand is a 16 x 16 identity; the MMA of K chunk kc targets only the 16 accumulator columns of that
    //          chunk's channels.  The centre view of the halo tile is the A operand: no global residual read.
    //          Only 2 x 16 x 16 B of IDENT_BYTES are used; the region stays larger on purpose (see launch_t).
    constexpr int IDENT_BYTES = 2 * (2 * N - 16) * 16;
    __half* ones = reinterpret_cast<__half*>(smem + (size_t)NST * stage_bytes + 1024 + 256 + N * sizeof(float));
    __half* biasB = ones + 2 * 128 * 8;
    __half* ident = biasB + 2 * N * 8;
    uint8_t* wres = smem + (((size_t)NST * stage_bytes + 1024 + 256 + N * sizeof(float) + 2 * 128 * 16 + 2 * N * 16 + IDENT_BYTES + 127) & ~(size_t)127);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_img = a.tiles_x * a.tiles_y;
    const int ntiles = tiles_img * a.batch;  // image-major: tile -> (image, ty, tx)
    const int KCP = a.Cin / 16;                    // K chunks per parity sub-image (all of them for stride 1)
    const int KC = TAPS == 9 ? KCP : (TAPS == 5 ? 5 * KCP : 4 * KCP);
    const uint32_t dskip = (uint32_t)(a.dbg_skip * KC);  // diagnostics: first recorded pipeline iteration

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < NST; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 8); }
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = threadIdx.x; i < N; i += NTHREADS) {
        // conv: GEMM column = output channel; deconv: column = parity * ocs + channel
        const int ch = a.epi == TC_EPI_DECONV ? (a.ocs > 0 ? i % a.ocs : i) : i;
        slope_s[i] = (a.act_mode == 1 ? a.slope : ((a.act_mode == 2 && ch < a.Cout) ? a.prelu[ch] : 1.f)) - 1.f;  // stored as slope - 1
    }
    for (int i = threadIdx.x; i < 2 * 128 * 8; i += NTHREADS) ones[i] = __float2half_rn((i < 128 * 8 && (i & 7) < 3) ? 1.f : 0.f);
    for (int i = threadIdx.x; i < 2 * N; i += NTHREADS) {
        const int n = i % N, hf = i / N;
        uint4 z = make_uint4(0, 0, 0, 0);
        if (hf == 0) {
            const float b = a.bias[n];
            const __half h0 = __float2half_rn(b);
            const float r1 = b - __half2float(h0);
            const __half h1 = __float2half_rn(r1);
            const __half h2 = __float2half_rn(r1 - __half2float(h1));
            z.x = pack2(h0, h1);
            z.y = pack2(h2, __float2half_rn(0.f));
        }
        *reinterpret_cast<uint4*>(biasB + (size_t)i * 8) = z;
    }
    if (a.res_mode == 3) {
        // 16 x 16 identity [half][16 rows][8]
        for (int i = threadIdx.x; i < 2 * 16 * 8; i += NTHREADS) {
            const int j = i & 7, r = (i >> 3) & 15, hf = i >> 7;
            ident[i] = __float2half_rn(r == hf * 8 + j ? 1.f : 0.f);
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the tensor core
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    unsigned long long* dbg = a.dbg ? a.dbg + (size_t)blockIdx.x * 64 : nullptr;
    if (dbg && threadIdx.x == 0) {
        dbg[0] = clock64();
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        dbg[60] = gt;
    }

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t it = 0;
            int s = 0;
            uint32_t ph = 0;
            if (a.wres) {
                mbar_arrive_expect_tx(wbar, (uint32_t)(KC * W_BYTES));
                for (int kc = 0; kc < KC; kc++) bulk_load_1d(wres + (size_t)kc * W_BYTES, a.wpk + (size_t)kc * (W_BYTES / 2), W_BYTES, wbar);
            }
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const int bimg = tile / tiles_img, trem = tile - bimg * tiles_img;
                const int tx = trem % a.tiles_x, ty = trem / a.tiles_x;
                const int x0 = tx * TVALID, y0 = ty * (2 * MT);
                for (int kc = 0, q = 0; kc < KC; kc++, it++) {
                    if (q == 0) {
                        mbar_wait(&empty[s], ph ^ 1);
                        mbar_arrive_expect_tx(&full[s], (uint32_t)(KS * (A_PLANE * nplanes + (a.wres ? 0 : W_BYTES))));
                    }
                    uint8_t* st = smem + (size_t)s * stage_bytes + (size_t)q * sub_bytes;
                    for (int p = 0; p < nplanes; p++) {
                        if constexpr (TAPS == 5) tma_load_4d(st + p * A_PLANE, &tmA, &full[s], (x0 - 2) * 4, y0 - 2 + kc % 5, p * (2 * KCP) + 2 * (kc / 5), bimg);
                        else tma_load_4d(st + p * A_PLANE, &tmA, &full[s], (x0 - 1) * 4, y0 - 1, p * (2 * KC) + 2 * kc, bimg);  // 16 B per pixel = 4 u32 elements
                    }
                    if (!a.wres) bulk_load_1d(st + nplanes * A_PLANE, a.wpk + (size_t)kc * (W_BYTES / 2), W_BYTES, &full[s]);
                    if (dbg && it - dskip < 12u) dbg[1 + it - dskip] = clock64();
                    if (++q == KS) { q = 0; if (++s == NST) { s = 0; ph ^= 1; } }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: all 32 lanes run the loop convergently, one elected lane issues each instruction =====
        {
            const uint32_t idesc = (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // f16 x f16 -> f32, K-major A and B
            // descriptor words: lo = start>>4 | (LBO>>4)<<16 ; hi = SBO>>4 | version(1)<<14
            constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);
            constexpr uint32_t A_LBO = ((uint32_t)(ROWS * TWP * 16) >> 4) << 16;
            constexpr uint32_t B_LBO = ((uint32_t)(N * 16) >> 4) << 16;
            // (The weight-stationary form tcgen05.mma.ws -- the MT MMAs of a tap sharing one B fetch -- was measured and is
            // not used: same tile period as this plain form, see profiles/r1_epilogue/mma_ws_ab.txt.)
            uint32_t it = 0, tcount = 0;
            int s = 0;
            uint32_t ph = 0;
            if (a.wres) {
                mbar_wait(wbar, 0);
                tc_fence_after();
            }
            const uint32_t wres_addr = smem_u32(wres);
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, tcount++) {
                const int buf = tcount & 1;
                const uint32_t aph = (tcount >> 1) & 1;
                mbar_wait(&acc_empty[buf], aph ^ 1);
                tc_fence_after();
                const uint32_t acc0 = tmem_base + buf * ACC_COLS;
                {   // accumulator := bias (see `ones` / `biasB`)
                    const uint32_t o_lo = (smem_u32(ones) >> 4) | (((uint32_t)(128 * 16) >> 4) << 16);
                    const uint32_t bb_lo = (smem_u32(biasB) >> 4) | B_LBO;
#pragma unroll
                    for (int m = 0; m < MT; m++)
                        umma_f16_elect(acc0 + m * N, o_lo, DESC_HI, bb_lo, DESC_HI, idesc, 0u);
                }
                for (int kc = 0, q = 0; kc < KC; kc++, it++) {
                    if (q == 0) {
                        mbar_wait(&full[s], ph);
                        tc_fence_after();
                    }
                    if (dbg && it - dskip < 12u && lane == 0) dbg[16 + it - dskip] = clock64();
                    const uint32_t st = smem_u32(smem + (size_t)s * stage_bytes + (size_t)q * sub_bytes);
                    const uint32_t a_base = (st >> 4) | A_LBO;
                    const uint32_t b_base = ((a.wres ? wres_addr + (uint32_t)(kc * W_BYTES) : st + nplanes * A_PLANE) >> 4) | B_LBO;
                    constexpr int ROWSTEP16 = (2 * TWP * 16) >> 4;  // accumulator m+1 starts 2 tile rows further
                    if constexpr (TAPS == 5) {
#pragma unroll
                        for (int dx = 0; dx < 5; dx++) {  // the five taps of kernel row kc % 5
                            const uint32_t b_lo = b_base + (uint32_t)(dx * (2 * N * 16) >> 4);
                            const uint32_t a_lo = a_base + (uint32_t)dx;
                            if (nplanes == 2) umma_issue_tap<MT, 2, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                            else umma_issue_tap<MT, 1, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                        }
                    } else if constexpr (TAPS == 9 && tc_paired(N)) {
                        // Paired issue: the view of halo rows 2j, 2j+1 is the dy=0 operand of accumulator j AND the dy=2 operand of
                        // accumulator j-1, whose TMEM columns are adjacent -- one 2N-column MMA against [W_dy2 | W_dy0] replaces two
                        // N-column ones (A is fetched from shared memory once instead of twice; 2*MT+1 MMAs per kernel column instead
                        // of 3*MT).  Weight block of (kc, dx): [half][3N rows: dy2 | dy0 | dy1][8] (to_paired_layout).  res_mode 3
                        // adds the identity tap onto the 16 accumulator columns of this chunk's channels.  Every MMA of the chunk is
                        // issued from ONE asm block with literal operand offsets (tools/gen_mma_issue.py chunk_block).
                        constexpr uint32_t B3_LBO = ((uint32_t)(3 * N * 16) >> 4) << 16;
                        constexpr uint32_t idesc2 = (1u << 4) | ((uint32_t)((2 * N) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
                        constexpr uint32_t I16_LBO = ((uint32_t)(16 * 16) >> 4) << 16;
                        constexpr uint32_t idesc16 = (1u << 4) | ((uint32_t)(16 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
                        const uint32_t b_addr = a.wres ? wres_addr + (uint32_t)(kc * W_BYTES) : st + nplanes * A_PLANE;
                        const uint32_t b_lo = (b_addr >> 4) | B3_LBO;
                        const uint32_t id_lo = (smem_u32(ident) >> 4) | I16_LBO;
                        const uint32_t id_on = a.res_mode == 3 ? 1u : 0u;
                        if (nplanes == 2) umma_issue_chunk_paired<N, MT, 2>(acc0, a_base, b_lo, DESC_HI, idesc, idesc2, id_on, id_lo, idesc16, acc0 + (uint32_t)(16 * kc));
                        else umma_issue_chunk_paired<N, MT, 1>(acc0, a_base, b_lo, DESC_HI, idesc, idesc2, id_on, id_lo, idesc16, acc0 + (uint32_t)(16 * kc));
                    } else if constexpr (TAPS == 9) {
                        // 2N > 256 (N = 192): nine N-column taps over [tap][half][N][8] weights; the launcher never selects the
                        // identity tap for these layers
#pragma unroll
                        for (int tap = 0; tap < 9; tap++) {
                            const int dy = tap / 3, dx = tap - dy * 3;
                            const uint32_t b_lo = b_base + (uint32_t)(tap * (2 * N * 16) >> 4);
                            const uint32_t a_lo = a_base + (uint32_t)(((dy * TWP + dx) * 16) >> 4);
                            if (nplanes == 2) umma_issue_tap<MT, 2, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                            else umma_issue_tap<MT, 1, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                        }
                    } else {
                        const int par = kc / KCP, py = par >> 1, px = par & 1;
#pragma unroll
                        for (int iy = 0; iy < 2; iy++)
#pragma unroll
                            for (int ix = 0; ix < 2; ix++) {
                                if (iy > py || ix > px) continue;  // even sub-images contribute one tap per axis (uniform branch)
                                // odd sub-image: slot 0 = tap d=0 (previous row/col, view offset 0), slot 1 = tap d=2 (view offset 1)
                                // even sub-image: single slot = tap d=1 (view offset 1)
                                const int oy = py ? iy : 1, ox = px ? ix : 1;
                                const uint32_t b_lo = b_base + (uint32_t)((iy * 2 + ix) * (2 * N * 16) >> 4);
                                const uint32_t a_lo = a_base + (uint32_t)(((oy * TWP + ox) * 16) >> 4);
                                if (nplanes == 2) umma_issue_tap<MT, 2, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                                else umma_issue_tap<MT, 1, (A_PLANE >> 4), ROWSTEP16, N>(acc0, a_lo, b_lo, DESC_HI, idesc, 1u);
                            }
                    }
                    if (q == KS - 1) umma_commit_elect(&empty[s]);  // frees the stage once the MMAs above have read it
                    if (dbg && it - dskip < 12u && lane == 0) dbg[32 + it - dskip] = clock64();
                    if (++q == KS) { q = 0; if (++s == NST) { s = 0; ph ^= 1; } }
                }
                umma_commit_elect(&acc_full[buf]);
            }
        }
    } else {
        // ===== epilogue warps =====
        // Per tile the accumulators are drained in NBLK blocks of CB channels.  The residual (16 B per 8-channel group
        // and plane) for block b+1 is fetched into registers while block b is converted and stored, and the fetch for
        // the first block is issued before waiting for the MMAs, so global-memory latency overlaps the tensor work.
        constexpr int CB = (N % 32 == 0) ? 32 : ((N % 48 == 0) ? 48 : 16);
        constexpr int NCB = N / CB, NBLK = MT * NCB, G = CB / 8;
        const int q = warp & 3;  // TMEM lane quarter this warp may access
        const int ehalf = (warp - 2) >> 2;  // the two warps of a quarter take alternate channel blocks
        const int p = q * 32 + lane;  // flattened position inside an accumulator
        const int xr = p & (TWP - 1), yrow = p >> 6;
        uint32_t tcount = 0;
        const size_t HW = (size_t)a.H * a.W;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, tcount++) {
            const int buf = tcount & 1;
            const uint32_t aph = (tcount >> 1) & 1;
            const int bimg = tile / tiles_img, trem = tile - bimg * tiles_img;
            const int tx = trem % a.tiles_x, ty = trem / a.tiles_x;
            const int x0 = tx * TVALID, y0 = ty * (2 * MT);
            const int x = x0 + xr;
            const __half* res_b = a.res + (size_t)bimg * a.res_bstride;
            __half* out_b = a.out + (size_t)bimg * a.out_bstride;
            float* outf_b = a.out_f32 + (size_t)bimg * a.outf_bstride;
            const bool xvalid = xr < TVALID && x < a.W;
            if (a.epi == TC_EPI_C8 && (a.res_mode == 0 || a.res_mode == 3) && a.act_mode != 2) {
                // No residual to fetch (none, or already added by the identity tap), bias already in the accumulator,
                // one slope for all channels: v = leaky(acc) on packed fp32 pairs, nothing but registers between the TMEM
                // load and the store.  Loads are software pipelined one block (CBL channels x 32 positions) ahead.
                constexpr int CBL = (N % 32 == 0) ? 32 : 16;
                constexpr int NCBL = N / CBL, NBLKL = MT * NCBL;
                const float sm1 = a.act_mode == 1 ? a.slope - 1.f : 0.f;
                const float2 sm1v = make_float2(sm1, sm1);
                // per-thread output address pieces: block (m, cb) -> obase + m * mstep + cb * cbstep
                const bool s2d = a.out_s2d != 0;
                const int yb = y0 + yrow;  // row of accumulator 0; accumulator m is 2 rows further down each
                const size_t cg_stride = !s2d ? HW : (HW >> 2);
                const size_t pix0 = !s2d ? (size_t)yb * a.W + x : (size_t)(yb >> 1) * (a.W >> 1) + (x >> 1);
                const size_t cg_base = !s2d ? 0 : (size_t)((yb & 1) * 2 + (x & 1)) * a.out_cgroups;
                __half* const obase = out_b + (cg_base * cg_stride + pix0) * 8;
                const size_t mstep = (!s2d ? (size_t)2 * a.W : (size_t)(a.W >> 1)) * 8;
                const size_t cbstep = (size_t)(CBL / 8) * cg_stride * 8, gstep = cg_stride * 8;
                auto ldblk = [&](int blk, uint32_t* r) {
                    const int m = blk / NCBL, cb = blk - m * NCBL;
                    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + buf * ACC_COLS + m * N + cb * CBL;
                    if constexpr (CBL == 32) tmem_ld32(trow, r);
                    else tmem_ld16(trow, r);
                };
                auto waitblk = [&](uint32_t* r) {
                    if constexpr (CBL == 32) tmem_ld_wait_dep32(r);
                    else tmem_ld_wait_dep16(r);
                };
                auto stblk = [&](int blk, const uint32_t* r, auto split_tag) {
                    constexpr bool SPLIT = decltype(split_tag)::value;
                    const int m = blk / NCBL, cb = blk - m * NCBL;
                    if (!(xvalid && yb + 2 * m < a.H)) return;
                    __half* const op = obase + m * mstep + cb * cbstep;
#pragma unroll
                    for (int g = 0; g < CBL / 8; g++) {
                        uint32_t hw_[4], lw_[4];
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            float2 v = make_float2(__uint_as_float(r[g * 8 + 2 * k]), __uint_as_float(r[g * 8 + 2 * k + 1]));
                            // leaky / identity: v*s for v < 0  ==  v + min(v,0)*(s-1)
                            v = __ffma2_rn(make_float2(fminf(v.x, 0.f), fminf(v.y, 0.f)), sm1v, v);
                            const __half2 h = __float22half2_rn(v);
                            hw_[k] = *reinterpret_cast<const uint32_t*>(&h);
                            if constexpr (SPLIT) {
                                const float2 f = __half22float2(h);
                                const __half2 l = __floats2half2_rn(v.x - f.x, v.y - f.y);
                                lw_[k] = *reinterpret_cast<const uint32_t*>(&l);
                            }
                        }
                        *reinterpret_cast<uint4*>(op + g * gstep) = make_uint4(hw_[0], hw_[1], hw_[2], hw_[3]);
                        if constexpr (SPLIT) *reinterpret_cast<uint4*>(op + a.out_plane + g * gstep) = make_uint4(lw_[0], lw_[1], lw_[2], lw_[3]);
                    }
                };
                auto stsel = [&](int blk, const uint32_t* r) {
                    if (a.split_out) stblk(blk, r, std::true_type{});
                    else stblk(blk, r, std::false_type{});
                };
                uint32_t ra[CBL], rb[CBL];
                mbar_wait(&acc_full[buf], aph);
                tc_fence_after();
                if (dbg && warp == 2 && lane == 0 && tcount - (uint32_t)a.dbg_skip < 4u) dbg[44 + 2 * (tcount - a.dbg_skip)] = clock64();
                if (ehalf < NBLKL) {
                    ldblk(ehalf, ra);
#pragma unroll 1
                    for (int blk = ehalf; blk < NBLKL; blk += 4) {
                        waitblk(ra);
                        if (blk + 2 < NBLKL) ldblk(blk + 2, rb);
                        stsel(blk, ra);
                        if (blk + 2 < NBLKL) {
                            waitblk(rb);
                            if (blk + 4 < NBLKL) ldblk(blk + 4, ra);
                            stsel(blk + 2, rb);
                        }
                    }
                }
            } else if (a.epi == TC_EPI_C8) {
                // v = act(acc + bias + m1*res) + m2*res with per-channel slopes from shared memory: one branch-free body
                // for every (residual, leaky / PReLU / none) combination keeps the unrolled code small (an earlier, fully
                // unrolled and flag-branchy version was 215 KB of SASS and instruction-fetch bound).
                const float m1 = a.res_mode == 1 ? 1.f : 0.f, m2 = a.res_mode == 2 ? 1.f : 0.f;
                const bool has_res = a.res_mode != 0;
                auto prefetch = [&](int blk, uint4* dst) {
                    const int m = blk / NCB, cb = blk % NCB;
                    const int y = y0 + 2 * m + yrow;
                    if (!has_res || !xvalid || y >= a.H) return;
#pragma unroll
                    for (int g = 0; g < G; g++) {
                        const size_t off = ((size_t)(cb * G + g) * HW + (size_t)y * a.W + x) * 8;
                        dst[g] = __ldg(reinterpret_cast<const uint4*>(res_b + off));
                        if (a.res_split) dst[G + g] = __ldg(reinterpret_cast<const uint4*>(res_b + a.res_plane + off));
                    }
                };
                auto process = [&](int blk, const uint4* rcur) {
                    const int m = blk / NCB, cb = blk % NCB;
                    const int y = y0 + 2 * m + yrow;
                    const bool valid = xvalid && y < a.H;
                    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + buf * ACC_COLS + m * N + cb * CB;
                    const size_t pix = !a.out_s2d ? (size_t)y * a.W + x : (size_t)(y >> 1) * (a.W >> 1) + (x >> 1);
                    const size_t cg_stride = !a.out_s2d ? HW : (HW >> 2);
                    const size_t cg_base = !a.out_s2d ? 0 : (size_t)((y & 1) * 2 + (x & 1)) * a.out_cgroups;
#pragma unroll
                    for (int c = 0; c < CB / 16; c++) {
                        uint32_t r[16];
                        tmem_ld16(trow + c * 16, r);
                        tmem_ld_wait();
                        if (valid) {
#pragma unroll
                            for (int g2 = 0; g2 < 2; g2++) {
                                const int gl = c * 2 + g2;   // group inside the block
                                const int cg = cb * G + gl;  // global 8-channel group
                                const float4 sA = *reinterpret_cast<const float4*>(slope_s + cg * 8), sB = *reinterpret_cast<const float4*>(slope_s + cg * 8 + 4);
                                const float ss[8] = {sA.x, sA.y, sA.z, sA.w, sB.x, sB.y, sB.z, sB.w};  // slope - 1
                                float v[8], rr[8];
#pragma unroll
                                for (int j = 0; j < 8; j++) { v[j] = __uint_as_float(r[g2 * 8 + j]); rr[j] = 0.f; }  // bias: already in the accumulator
                                if (has_res) {
                                    const __half2* hh = reinterpret_cast<const __half2*>(&rcur[gl]);
#pragma unroll
                                    for (int k = 0; k < 4; k++) { float2 f = __half22float2(hh[k]); rr[2 * k] = f.x; rr[2 * k + 1] = f.y; }
                                    if (a.res_split) {
                                        const __half2* ll = reinterpret_cast<const __half2*>(&rcur[G + gl]);
#pragma unroll
                                        for (int k = 0; k < 4; k++) { float2 f = __half22float2(ll[k]); rr[2 * k] += f.x; rr[2 * k + 1] += f.y; }
                                    }
#pragma unroll
                                    for (int j = 0; j < 8; j++) v[j] = fmaf(m1, rr[j], v[j]);
                                }
                                // leaky / PReLU / identity: v*s for v < 0  ==  v + min(v,0)*(s-1)
#pragma unroll
                                for (int j = 0; j < 8; j++) v[j] = fmaf(fminf(v[j], 0.f), ss[j], v[j]);
                                if (has_res) {
#pragma unroll
                                    for (int j = 0; j < 8; j++) v[j] = fmaf(m2, rr[j], v[j]);
                                }
                                __half2 h[4];
#pragma unroll
                                for (int k = 0; k < 4; k++) h[k] = __floats2half2_rn(v[2 * k], v[2 * k + 1]);
                                const size_t ooff = ((cg_base + cg) * cg_stride + pix) * 8;
                                *reinterpret_cast<uint4*>(out_b + ooff) = make_uint4(*reinterpret_cast<uint32_t*>(&h[0]), *reinterpret_cast<uint32_t*>(&h[1]),
                                                                                     *reinterpret_cast<uint32_t*>(&h[2]), *reinterpret_cast<uint32_t*>(&h[3]));
                                if (a.split_out) {
                                    __half2 l[4];
#pragma unroll
                                    for (int k = 0; k < 4; k++) {
                                        float2 f = __half22float2(h[k]);
                                        l[k] = __floats2half2_rn(v[2 * k] - f.x, v[2 * k + 1] - f.y);
                                    }
                                    *reinterpret_cast<uint4*>(out_b + a.out_plane + ooff) = make_uint4(*reinterpret_cast<uint32_t*>(&l[0]), *reinterpret_cast<uint32_t*>(&l[1]),
                                                                                                       *reinterpret_cast<uint32_t*>(&l[2]), *reinterpret_cast<uint32_t*>(&l[3]));
                                }
                            }
                        }
                    }
                };
                uint4 rb0[2 * G], rb1[2 * G];
                // this warp's blocks: ehalf, ehalf + 2, ehalf + 4, ...
                if (ehalf < NBLK) prefetch(ehalf, rb0);
                mbar_wait(&acc_full[buf], aph);
                tc_fence_after();
                if (dbg && warp == 2 && lane == 0 && tcount - (uint32_t)a.dbg_skip < 4u) dbg[44 + 2 * (tcount - a.dbg_skip)] = clock64();
#pragma unroll 1
                for (int blk = ehalf; blk < NBLK; blk += 4) {
                    if (blk + 2 < NBLK) prefetch(blk + 2, rb1);
                    process(blk, rb0);
                    if (blk + 2 < NBLK) {
                        if (blk + 4 < NBLK) prefetch(blk + 4, rb0);
                        process(blk + 2, rb1);
                    }
                }
            } else {
                // deconv4x4s2 (+ optional PixelShuffle r) epilogue: column n = parity * ocs + oc, parity = py*2+px.
                // deconv output pixel (2y+py, 2x+px), channel oc; PixelShuffle(r): oc = qq*r*r + sh*r + sw lands at
                // row (2y+py)*r+sh, column (2x+px)*r+sw of plane qq -> for fixed (qq, sh, py) the 2r columns
                // 2r*x .. 2r*x+2r-1 are contiguous: one 16-byte (r=2) / 8-byte (r=1) store per thread, coalesced per warp.
                mbar_wait(&acc_full[buf], aph);
                tc_fence_after();
                if constexpr (N <= 96) {
                const int r_ = a.ps;
                const int OH = a.H * 2 * r_, OW = a.W * 2 * r_;
                if (N == 96 && r_ == 2 && a.act_mode == 0 && a.out_planes == 5) {
                    // the IFNet flow head (24 channels -> PixelShuffle(2) -> 4 flow + 1 mask planes, the sixth plane is never
                    // read): per (accumulator m, output-row parity py) 2 x 20 of the 48 columns are needed; they go out
                    // as 10 coalesced 16-byte stores straight from the loaded registers.  The bias is already in the accumulator.
                    constexpr int OCS = 24, NH = 48, NIT = 2 * MT;
                    auto ld = [&](int it, uint32_t* r) {
                        const uint32_t t = tmem_base + ((uint32_t)(q * 32) << 16) + buf * ACC_COLS + (it >> 1) * N + (it & 1) * NH;
                        tmem_ld16(t, r); tmem_ld4(t + 16, r + 16);                  // px = 0: oc 0..19
                        tmem_ld16(t + OCS, r + 20); tmem_ld4(t + OCS + 16, r + 36);  // px = 1: oc 0..19
                    };
                    auto wt = [&](uint32_t* r) { tmem_ld_wait_dep32(r); tmem_ld_wait_dep16(r + 24); };  // one wait; 40 of the registers named
                    auto stv = [&](int it, const uint32_t* r) {
                        const int m = it >> 1, py = it & 1;
                        const int y = y0 + 2 * m + yrow;
                        if (!(xvalid && y < a.H)) return;
                        float* o = outf_b + (size_t)((2 * y + py) * 2) * OW + 4 * x;
#pragma unroll
                        for (int qq = 0; qq < 5; qq++)
#pragma unroll
                            for (int sh = 0; sh < 2; sh++) {
                                const int o0 = qq * 4 + sh * 2;
                                *reinterpret_cast<float4*>(o + ((size_t)qq * OH + sh) * OW) =
                                    make_float4(__uint_as_float(r[o0]), __uint_as_float(r[o0 + 1]), __uint_as_float(r[20 + o0]), __uint_as_float(r[20 + o0 + 1]));
                            }
                    };
                    uint32_t ra[40];
#pragma unroll 1
                    for (int it = ehalf; it < NIT; it += 2) {
                        ld(it, ra);
                        wt(ra);
                        stv(it, ra);
                    }
                } else
#pragma unroll 1
                for (int m = ehalf; m < MT; m += 2) {
                    const int y = y0 + 2 * m + yrow;
                    const bool valid = xvalid && y < a.H;
                    const uint32_t trow = tmem_base + ((uint32_t)(q * 32) << 16) + buf * ACC_COLS + m * N;
                    constexpr int OCS = N / 4, NH = N / 2;
                    // the two output-row parities are independent halves of the columns: halves the live registers
#pragma unroll
                    for (int py = 0; py < 2; py++) {
                        float v[NH];
#pragma unroll
                        for (int c0 = 0; c0 < NH; c0 += 16) {
                            uint32_t r[16];
                            tmem_ld16(trow + py * NH + c0, r);
                            tmem_ld_wait();
#pragma unroll
                            for (int j = 0; j < 16; j++) {
                                float val = __uint_as_float(r[j]);  // bias: already in the accumulator
                                if (a.act_mode == 3) val = 1.f / (1.f + expf(-fminf(fmaxf(val, -88.3762626647949f), 88.3762626647949f)));
                                else if (a.act_mode != 0) val = fmaf(fminf(val, 0.f), slope_s[py * NH + c0 + j], val);  // leaky / PReLU: v + min(v, 0) * (slope - 1)
                                v[c0 + j] = val;
                            }
                        }
                        if (!valid) continue;
                        if (r_ == 2) {
#pragma unroll
                            for (int oc4 = 0; oc4 < OCS / 4; oc4++) {  // oc4 = qq
                                if (oc4 * 4 >= a.Cout || (a.out_planes > 0 && oc4 >= a.out_planes)) break;
#pragma unroll
                                for (int sh = 0; sh < 2; sh++) {
                                    const int o0 = oc4 * 4 + sh * 2;  // oc for sw = 0
                                    float4 w4 = make_float4(v[o0], v[o0 + 1], v[OCS + o0], v[OCS + o0 + 1]);  // px = 0 | px = 1
                                    const int oy = (2 * y + py) * 2 + sh;
                                    *reinterpret_cast<float4*>(outf_b + ((size_t)oc4 * OH + oy) * OW + 4 * x) = w4;
                                }
                            }
                        } else {
#pragma unroll
                            for (int oc = 0; oc < OCS; oc++) {
                                if (oc >= a.Cout) break;
                                float2 w2 = make_float2(v[oc], v[OCS + oc]);
                                *reinterpret_cast<float2*>(outf_b + ((size_t)oc * OH + 2 * y + py) * OW + 2 * x) = w2;
                            }
                        }
                    }
                }
                }  // N <= 96 (deconv instances)
            }
            tc_fence_before();
            __syncwarp();
            if (dbg && warp == 2 && lane == 0 && tcount - (uint32_t)a.dbg_skip < 4u) dbg[45 + 2 * (tcount - a.dbg_skip)] = clock64();
            if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (dbg && threadIdx.x == 0) dbg[56] = clock64();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess) return nullptr;
    fn = (EncodeTiledFn)p;
    return fn;
}

template <int N, int MT, int STAGES, int TAPS>
static int launch_t(const TcConvArgs& a_in, const CUtensorMap& tm, cudaStream_t st) {
    TcConvArgs a = a_in;
    constexpr int TWP = 64;
    constexpr int ROWS = TAPS == 5 ? 2 * MT : 2 * MT + 2;
    constexpr int A_PLANE = 2 * ROWS * TWP * 16;
    constexpr int W_BYTES = TAPS * 2 * N * 16;
    const int nplanes = a.split_in ? 2 : 1;
    // barriers etc. (256) + slope_s + ones tile (4 KB) + bias B matrix + identity matrix (res_mode 3, or resident weights)
    const size_t consts = 1024 + 256 + N * sizeof(float) + 2 * 128 * 16 + (size_t)2 * N * 16;
    // The identity tap uses 512 B of this; shrinking the reservation would change stages / ks of some layers (to be measured).
    const size_t ident_bytes = (size_t)2 * (2 * N - 16) * 16;
    // resident weights (stride-1 kernels): the whole packed layer next to activation-only stages, when it fits
    const size_t w_all = (size_t)(a.Cin / 16) * W_BYTES * (TAPS == 5 ? 5 : 1);
    const size_t budget = 227 * 1024;
    const size_t stage_a = (size_t)((A_PLANE * nplanes + 1023) & ~1023), stage_aw = (size_t)((A_PLANE * nplanes + W_BYTES + 1023) & ~1023);
    // resident weights need at least STAGES activation-only stages next to the whole layer
    a.wres = TAPS == 9 && ((STAGES * stage_a + consts + ident_bytes + 127) & ~(size_t)127) + w_all <= budget;
    // chunks per pipeline stage: resident-weight kernels only, KC divisible, >= 2 stages left
    const size_t fixed = a.wres ? consts + ident_bytes + 127 + w_all : consts + (a.res_mode == 3 ? ident_bytes : 0);
    a.ks = 1;
    if (a.wres && (a.Cin / 16) % TC_KS_DEFAULT == 0 && (budget - fixed) / (stage_a * TC_KS_DEFAULT) >= 2) a.ks = TC_KS_DEFAULT;
    const int stage_bytes = (int)(a.wres ? stage_a * a.ks : stage_aw);
    // pipeline depth: what shared memory allows (the stages are what hides the L2 / HBM latency of the activation tiles)
    int nst = (int)((budget - fixed) / stage_bytes);
    if (nst > 8) nst = 8;
    if (nst < STAGES && a.ks == 1) nst = STAGES;
    a.stages = nst;
    const size_t smem = a.wres ? (((size_t)nst * stage_bytes + consts + ident_bytes + 127) & ~(size_t)127) + w_all : (size_t)nst * stage_bytes + fixed;
    if (smem > 227 * 1024) return -2;
    // the attribute is per device: one process may drive several GPUs (src/main.cpp -g 0,1,...)
    static size_t configured[64] = {};
    static std::mutex configured_mu;  // lanes of several engines / threads may launch the same instantiation for the first time together
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) return -3;
    {
        std::lock_guard<std::mutex> lk(configured_mu);
        if (smem > configured[dev]) {
            if (cudaFuncSetAttribute(tc_conv3x3_kernel<N, MT, STAGES, TAPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return -3;
            configured[dev] = smem;
        }
    }
    int ntiles = a.tiles_x * a.tiles_y * a.batch;
    int grid = ntiles < a.num_sms ? ntiles : a.num_sms;
    tc_conv3x3_kernel<N, MT, STAGES, TAPS><<<grid, NTHREADS, smem, st>>>(tm, a);
    g_launch_count++;
    return 0;
}

int tc_conv_tile_rows(int N) { return N <= 64 ? 8 : (N <= 128 ? 4 : 2); }  // 2 * MT

template <int N, int MT, int STAGES>
static int launch_n(const TcConvArgs& a, const CUtensorMap& tm, cudaStream_t st) {
    if constexpr (N == 48 || N == 96 || N == 128 || N == 192) {  // the widths of the 5x5 residual blocks (rife / HD / UHD / anime flownets)
        if (a.k5) return launch_t<N, MT, 2, 5>(a, tm, st);
    }
    if (a.k5) return -6;
    return a.s2 ? launch_t<N, MT, STAGES, 4>(a, tm, st) : launch_t<N, MT, STAGES, 9>(a, tm, st);
}

int launch_tc_conv(TcConvArgs a, const void* in, cudaStream_t st) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return -1;
    if (a.Cin % 16 || a.N % 16 || a.N < 16 || a.N > 256) return -4;
    const int nplanes = a.split_in ? 2 : 1;
    const int MT = tc_conv_tile_rows(a.N) / 2;
    if (a.k5 && (a.s2 || a.epi != TC_EPI_C8)) return -4;
    const int TWP = 64, TVALID = TWP - (a.k5 ? 4 : 2), tile_rows = 2 * MT;
    a.tiles_x = (a.W + TVALID - 1) / TVALID;
    a.tiles_y = (a.H + tile_rows - 1) / tile_rows;
    if (!a.num_sms) a.num_sms = 148;
    // activation tensor viewed as [planes * C/8][H][W*4] 32-bit words (16 B = one pixel's 8 channels)
    CUtensorMap tm;
    // stride 2: the input is the space-to-depth tensor, 4 sub-images of (H, W) = output size, Cin channels each
    const int cgroups = (a.s2 ? 4 : 1) * (a.Cin / 8);
    if (a.out_s2d && ((a.H | a.W) & 1)) return -7;
    if (a.batch < 1) a.batch = 1;
    if (a.out_cgroups <= 0) a.out_cgroups = a.Cout / 8;  // a launch that writes a channel slice of a wider tensor sets it to the tensor's groups
    if (a.res_mode == 3) return -9;  // internal value, selected below
    // residual == the conv's own input (the ResConv blocks): let the tensor core add it (identity tap, see the kernel)
    if (a.res_mode == 1 && a.epi == TC_EPI_C8 && !a.s2 && !a.k5 && a.res == (const __half*)in && a.Cin == a.N && a.Cout == a.N && a.N <= 128 && (!a.res_split) == (!a.split_in) &&
        (!a.split_in || a.res_plane == (size_t)a.Cin * a.H * a.W) && (a.batch == 1 || a.res_bstride == a.in_bstride))
        a.res_mode = 3;
    const size_t img_bytes = (size_t)nplanes * cgroups * a.H * a.W * 16;
    if (a.batch > 1 && a.in_bstride * 2 < img_bytes) return -8;
    cuuint64_t dims[4] = {(cuuint64_t)a.W * 4, (cuuint64_t)a.H, (cuuint64_t)nplanes * cgroups, (cuuint64_t)a.batch};
    cuuint64_t strides[3] = {(cuuint64_t)a.W * 16, (cuuint64_t)a.H * a.W * 16, a.batch > 1 ? (cuuint64_t)a.in_bstride * 2 : (cuuint64_t)img_bytes};
    cuuint32_t box[4] = {(cuuint32_t)(TWP * 4), (cuuint32_t)(a.k5 ? tile_rows : tile_rows + 2), 2, 1};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(&tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<void*>(in), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return -5;
    switch (a.N) {
        case 16: return launch_n<16, 4, 4>(a, tm, st);
        case 32: return launch_n<32, 4, 4>(a, tm, st);
        case 48: return launch_n<48, 4, 3>(a, tm, st);
        case 64: return launch_n<64, 4, 3>(a, tm, st);
        case 96: return launch_n<96, 2, 3>(a, tm, st);
        case 128: return launch_n<128, 2, 3>(a, tm, st);
        case 192: return launch_n<192, 1, 3>(a, tm, st);
        default: return -6;
    }
}

// ---- layout conversion kernels -------------------------------------------------------------------
// planar fp32 [C][H][W] -> C8 planar fp16 hi (+lo); channels are zero padded to Cpad (multiple of 8).
// s2d: space-to-depth variant [py*2+px][Cpad/8][H/2][W/2][8] feeding the stride-2 tensor-core conv.
__global__ void planar_to_c8_kernel(const float* __restrict__ in, __half* __restrict__ out, int C, int Cpad, int H, int W, int split, int s2d, size_t plane) {
    size_t HW = (size_t)H * W;
    size_t n = (size_t)(Cpad / 8) * HW;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    size_t cg = i / HW, pix = i - cg * HW;
    __half hi[8], lo[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
        int c = (int)cg * 8 + j;
        float v = c < C ? in[(size_t)c * HW + pix] : 0.f;
        hi[j] = __float2half_rn(v);
        lo[j] = __float2half_rn(v - __half2float(hi[j]));
    }
    size_t o = i;
    if (s2d) {
        int y = (int)(pix / W), x = (int)(pix - (size_t)y * W);
        o = (((size_t)((y & 1) * 2 + (x & 1)) * (Cpad / 8) + cg) * (H >> 1) + (y >> 1)) * (size_t)(W >> 1) + (x >> 1);
    }
    *reinterpret_cast<uint4*>(out + o * 8) = make_uint4(pack2(hi[0], hi[1]), pack2(hi[2], hi[3]), pack2(hi[4], hi[5]), pack2(hi[6], hi[7]));
    if (split) *reinterpret_cast<uint4*>(out + plane + o * 8) = make_uint4(pack2(lo[0], lo[1]), pack2(lo[2], lo[3]), pack2(lo[4], lo[5]), pack2(lo[6], lo[7]));
}
void launch_planar_to_c8(const float* in, __half* out, int C, int H, int W, int split, cudaStream_t st, int Cpad, int s2d) {
    if (Cpad <= 0) Cpad = (C + 7) / 8 * 8;
    size_t n = (size_t)(Cpad / 8) * H * W;
    planar_to_c8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, C, Cpad, H, W, split, s2d, (size_t)Cpad * H * W);
    g_launch_count++;
}
__global__ void c8_to_planar_kernel(const __half* __restrict__ in, float* __restrict__ out, int C, int Cpad, int H, int W, int split, int s2d, size_t plane) {
    size_t HW = (size_t)H * W;
    size_t n = (size_t)(Cpad / 8) * HW;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    size_t cg = i / HW, pix = i - cg * HW;
    size_t o = i;
    if (s2d) {
        int y = (int)(pix / W), x = (int)(pix - (size_t)y * W);
        o = (((size_t)((y & 1) * 2 + (x & 1)) * (Cpad / 8) + cg) * (H >> 1) + (y >> 1)) * (size_t)(W >> 1) + (x >> 1);
    }
    uint4 h = *reinterpret_cast<const uint4*>(in + o * 8);
    uint4 l = split ? *reinterpret_cast<const uint4*>(in + plane + o * 8) : make_uint4(0, 0, 0, 0);
    const __half* hh = reinterpret_cast<const __half*>(&h);
    const __half* ll = reinterpret_cast<const __half*>(&l);
#pragma unroll
    for (int j = 0; j < 8; j++) {
        int c = (int)cg * 8 + j;
        if (c < C) out[(size_t)c * HW + pix] = __half2float(hh[j]) + __half2float(ll[j]);
    }
}
void launch_c8_to_planar(const __half* in, float* out, int C, int H, int W, int split, cudaStream_t st, int Cpad, int s2d) {
    if (Cpad <= 0) Cpad = (C + 7) / 8 * 8;
    size_t n = (size_t)(Cpad / 8) * H * W;
    c8_to_planar_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(in, out, C, Cpad, H, W, split, s2d, (size_t)Cpad * H * W);
    g_launch_count++;
}

// ---- weight packing (host) -----------------------------------------------------------------------
// Paired MMA issue (tc_paired), for every stride-1 layer whose 2N fits one MMA.
// Measured (profiles/README.md, round-1 session 20): 16-channel mainloop stage of the 64->64 layer 2306 -> 1979 cycles,
// the layer itself 96.5 -> 84.2 us at 8 x 480x272, whole model 2195 -> 2311 frames/s at 1080p.
// [kc][tap = dy*3+dx][half][N][8] -> [kc][dx][half][3N rows: dy2 | dy0 | dy1][8]
static void to_paired_layout(std::vector<uint16_t>& w, int kcs, int N) {
    std::vector<uint16_t> o(w.size());
    static const int slot[3] = {1, 2, 0};  // row block of dy = 0, 1, 2
    for (int kc = 0; kc < kcs; kc++)
        for (int dy = 0; dy < 3; dy++)
            for (int dx = 0; dx < 3; dx++)
                for (int hf = 0; hf < 2; hf++)
                    for (int n = 0; n < N; n++) {
                        const size_t src = ((((size_t)kc * 9 + dy * 3 + dx) * 2 + hf) * N + n) * 8;
                        const size_t dst = ((((size_t)kc * 3 + dx) * 2 + hf) * (3 * N) + (size_t)slot[dy] * N + n) * 8;
                        for (int j = 0; j < 8; j++) o[dst + j] = w[src + j];
                    }
    w.swap(o);
}
// conv: w[oc][ic][3][3] fp32 (fp16-exact) -> wpk[kc][tap][half][n][8] fp16, n = oc (zero padded to N)
void pack_conv3x3_weights(const float* w, int cout, int cin, int N, std::vector<uint16_t>& out, int paired) {
    out.assign((size_t)(cin / 16) * 9 * 2 * N * 8, 0);
    for (int kc = 0; kc < cin / 16; kc++)
        for (int tap = 0; tap < 9; tap++)
            for (int hf = 0; hf < 2; hf++)
                for (int n = 0; n < cout; n++)
                    for (int j = 0; j < 8; j++) {
                        int ic = kc * 16 + hf * 8 + j;
                        __half h = __float2half_rn(w[((size_t)n * cin + ic) * 9 + tap]);
                        out[((((size_t)kc * 9 + tap) * 2 + hf) * N + n) * 8 + j] = __half_as_ushort(h);
                    }
    if (paired != 0 && tc_paired(N)) to_paired_layout(out, cin / 16, N);  // -1: what the launcher assumes; 1: paired where it fits
}
// conv 5x5 stride 1: w[oc][ic][5][5] fp32 (fp16-exact) -> wpk[kc][dy][dx][half][n][8]: one kernel row (five taps) per pipeline stage
void pack_conv5x5_weights(const float* w, int cout, int cin, int N, std::vector<uint16_t>& out) {
    out.assign((size_t)(cin / 16) * 25 * 2 * N * 8, 0);
    for (int kc = 0; kc < cin / 16; kc++)
        for (int tap = 0; tap < 25; tap++)
            for (int hf = 0; hf < 2; hf++)
                for (int n = 0; n < cout; n++)
                    for (int j = 0; j < 8; j++) {
                        int ic = kc * 16 + hf * 8 + j;
                        __half h = __float2half_rn(w[((size_t)n * cin + ic) * 25 + tap]);
                        out[((((size_t)kc * 25 + tap) * 2 + hf) * N + n) * 8 + j] = __half_as_ushort(h);
                    }
}
// conv 3x3 stride 2: w[oc][ic][3][3] -> wpk[4 parities][cinp/16][4 slots][2][N][8]; parity (py,px) of the space-to-depth
// input, slot (iy*2+ix) <-> tap dy = py ? 2*iy : 1, dx = px ? 2*ix : 1; input channels zero padded to cinp
void pack_conv3x3s2_weights(const float* w, int cout, int cin, int cinp, int N, std::vector<uint16_t>& out) {
    const int kcp = cinp / 16;
    out.assign((size_t)4 * kcp * 4 * 2 * N * 8, 0);
    for (int par = 0; par < 4; par++) {
        const int py = par >> 1, px = par & 1;
        for (int kc = 0; kc < kcp; kc++)
            for (int iy = 0; iy < (py ? 2 : 1); iy++)
                for (int ix = 0; ix < (px ? 2 : 1); ix++) {
                    const int dy = py ? 2 * iy : 1, dx = px ? 2 * ix : 1;
                    for (int hf = 0; hf < 2; hf++)
                        for (int n = 0; n < cout; n++)
                            for (int j = 0; j < 8; j++) {
                                int ic = kc * 16 + hf * 8 + j;
                                if (ic >= cin) continue;
                                __half h = __float2half_rn(w[((size_t)n * cin + ic) * 9 + dy * 3 + dx]);
                                out[(((((size_t)par * kcp + kc) * 4 + iy * 2 + ix) * 2 + hf) * N + n) * 8 + j] = __half_as_ushort(h);
                            }
                }
    }
}
// deconv 4x4 s2 p1: w[oc][ic][4][4] -> 3x3-neighbourhood GEMM with n = parity*ocs + oc:
// out(2y+py, 2x+px) = sum_{dy,dx} in(y-1+dy, x-1+dx) * w[oc][ic][3+py-2dy][3+px-2dx]  for dy-py, dx-px in {0,1}
void pack_deconv4x4_weights(const float* w, int cout, int cin, int ocs, int N, std::vector<uint16_t>& out, int paired) {
    out.assign((size_t)(cin / 16) * 9 * 2 * N * 8, 0);
    for (int kc = 0; kc < cin / 16; kc++)
        for (int dy = 0; dy < 3; dy++)
            for (int dx = 0; dx < 3; dx++)
                for (int par = 0; par < 4; par++) {
                    int py = par >> 1, px = par & 1;
                    if (dy - py < 0 || dy - py > 1 || dx - px < 0 || dx - px > 1) continue;
                    int ky = 3 + py - 2 * dy, kx = 3 + px - 2 * dx;
                    for (int hf = 0; hf < 2; hf++)
                        for (int oc = 0; oc < cout; oc++)
                            for (int j = 0; j < 8; j++) {
                                int ic = kc * 16 + hf * 8 + j;
                                __half h = __float2half_rn(w[((size_t)oc * cin + ic) * 16 + ky * 4 + kx]);
                                out[((((size_t)kc * 9 + dy * 3 + dx) * 2 + hf) * N + par * ocs + oc) * 8 + j] = __half_as_ushort(h);
                            }
                }
    if (paired != 0 && tc_paired(N)) to_paired_layout(out, cin / 16, N);
}

}  // namespace rife
