// libpifpaf_b200 -- backbone + heads forward for sm_100a.
//
// Replaces the cuDNN/ATen kernels behind the reference's torch.nn modules
// (paths relative to /root/reference/src/openpifpaf/):
//   Shell.forward                 network/nets.py:35-48
//   ShuffleNetV2K/InvertedResidualK   network/basenetworks.py:186-355
//   CompositeField4 (eval)        network/heads.py:330-378
//
// Activations are NHWC bf16 ("rows" = pixels, "columns" = channels).  Every 1x1
// convolution (97 % of the MACs of shufflenetv2k16) is one GEMM
//   out[M = B*H*W, N] = act[M, K] * W[N, K]^T,  f32 accumulate
// executed by k_gemm_tc: a persistent, warp-specialised tcgen05 kernel -- TMA
// (128B-swizzled tiles) -> shared-memory ring -> tcgen05.mma with the f32
// accumulator in TMEM (two accumulator stages) -> epilogue warps (tcgen05.ld,
// bias + ReLU, bf16) that also fuse torch.cat + channel_shuffle(2) (interleaving
// with the pass-through half) or the CompositeField4 eval epilogue (sigmoid,
// index-field add, softplus, f32 [B,F,comp,h,w] layout).
// Depthwise 5x5 and the 3-channel input conv are bandwidth-bound direct kernels.
#include <cuda.h>
#include <cuda_bf16.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <utility>
#include <vector>

#include "common.cuh"

namespace {

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                            int c0, int c1, int c2, int c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)),
          "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, bf16 inputs, f32 accumulate
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// the same, executed by a converged warp: descriptors as (lo, hi) words, one elected lane issues
__device__ __forceinline__ void umma_bf16_elect(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, e;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %2};\n\tmov.b64 db, {%3, %4};\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
        ::"r"(tmem_d), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred e;\n\t"
        "elect.sync _|e, 0xffffffff;\n\t"
        "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}"
        ::"r"(smem_u32(bar)) : "memory");
}
// mbarrier arrives when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// ---- thread-block cluster of two CTAs sharing the A operand (TMA multicast)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r;
}
// all threads of both CTAs
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// the box lands at the same shared-memory offset of every CTA in cta_mask and completes bytes on the mbarrier at
// the same offset there
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                               uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "h"(cta_mask), "r"(c0), "r"(c1)
        : "memory");
}
// arrives on the mbarrier at this offset in every CTA of cta_mask once the MMAs issued so far have completed
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}

// asynchronous TMEM load of 16 columns; results are valid only after tmem_ld_wait(v)
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr)
        : "memory");
}
// wait for all outstanding tcgen05.ld of this thread; the registers are in/out operands so that no use of them
// can be scheduled above the wait
__device__ __forceinline__ void tmem_ld_wait(uint32_t* v) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                   "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
                 :
                 : "memory");
}

// Programmatic dependent launch (PDL): a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may
// start while its predecessor in the stream is still draining; everything up to pdl_wait() (barrier init, TMEM
// allocation, descriptor prefetch, staging of constant weights / biases) overlaps the predecessor's tail.
// pdl_wait() returns once the predecessor has completed and its writes are visible -- it must precede every access
// to activations (reads AND writes: the predecessor may still be reading what this kernel overwrites).  Both are
// no-ops in a kernel launched the ordinary way.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ------------------------------------------------------------------ descriptors
constexpr int BM = 128;          // UMMA M (cta_group::1): TMEM lane == tile row
constexpr int BK = 64;           // one 128-byte swizzle atom of bf16 per smem row
constexpr int UMMA_K = 16;
constexpr int EPI_WARPS = 16;        // four warps per TMEM lane quadrant, each takes a quarter of the columns
constexpr int GEMM_THREADS = 64 + 32 * EPI_WARPS;   // warp 0 TMA, warp 1 MMA + TMEM alloc, warps 2..9 epilogue
constexpr int CHUNK = 16;        // epilogue column chunk (one tcgen05.ld.32x32b.x16)

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor):
// start>>4 | LBO(ignored for swizzled K-major)=1 @16 | SBO = 1024 B (8 rows x 128 B) >>4 @32 | version 1 @46 | layout 2 @61
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu);
    d |= static_cast<uint64_t>(1u) << 16;
    d |= static_cast<uint64_t>(1024u >> 4) << 32;
    d |= static_cast<uint64_t>(1u) << 46;
    d |= static_cast<uint64_t>(2u) << 61;
    return d;
}
// cute::UMMA::InstrDescriptor for kind::f16: c_format F32 (1) @4, a/b format BF16 (1) @7/@10,
// a/b K-major (0) @15/@16, N>>3 @17, M>>4 @24
__host__ __device__ inline uint32_t make_instr_desc(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
           (static_cast<uint32_t>(m >> 4) << 24);
}

// ------------------------------------------------------------------ GEMM arguments
enum { MODE_PLAIN = 0, MODE_SHUFFLE = 1, MODE_HEADS = 2, MODE_SCATTER = 3 };

// MODE_SCATTER: destination of one chunk of 16 GEMM columns (32 bytes per row, one 256-bit store per lane): base
// already points at the chunk's first column inside its tensor (a multiple of 16 channels)
struct DestGroup { __nv_bfloat16* base; int ld; int pad; };
static_assert(sizeof(DestGroup) == 16, "DestGroup is copied to shared memory as 16-byte entries");

// per GEMM output column (heads mode): plane = field * n_comp + comp; sub = (dy << 8) | dx is the PixelShuffle
// position of this conv channel inside the up x up block of its cell (heads.py:333-343), 0 without upsampling
struct HeadCol { int head; int plane; int op; int sub; };

struct GemmArgs {
    int M, N, K;                 // rows, real output channels, k extent (columns of the A view)
    int a_col0;                  // first column of the A view inside its tensor (TMA coordinate; multiple of 8)
    int block_n, n_blocks, m_blocks, num_k_blocks, stages;
    int mode, relu;              // relu: activation code (act_f)
    const float* bias;           // [n_blocks * block_n], zero padded
    // plain / shuffle
    __nv_bfloat16* out; int ldo; int out_col_off;
    const __nv_bfloat16* src0; int ld0; int src0_col_off; int half; int gap;
    int src_tma;                 // pass-through tile arrives by TMA in shared memory (else read from global)
    int b_resident;              // all K blocks of this CTA's weight tile stay in shared memory (loaded once)
    int pair, pair_stages;       // k_gemm_tc2 (CTA pairs, cta_group::2): on / ring depth per CTA
    int debug;                   // timing experiments only (PIFPAF_GEMM_DEBUG; results are wrong): 1 = no epilogue stores,
                                 // 2 = no MMAs issued, 4 = epilogue does not read TMEM, 8 = scatter pieces written as one row,
                                 // 16 = every scatter piece written as its own [pixels][width] tensor
    int mc;                      // weights-resident, two n blocks: the two CTAs of an M tile form a cluster and share A --
                                 // each loads one half (64 rows) of every A stage and multicasts it to both (tmap_src = the
                                 // 64-row A map); a stage is free when BOTH have consumed it
    // scatter: chunks of 16 columns go to different tensors (the 'bins' layout: every channel is written once,
    // into the buffer of the block that consumes it)
    const DestGroup* dest;       // [n_blocks * block_n / 16]
    // heads
    const HeadCol* head_cols;    // [n_blocks * block_n]
    float* head_base[4]; int head_planes[4];
    int hw, w;                   // pixels per image, field width (of the conv output)
    int up, up_low, out_h, out_w;   // PixelShuffle factor, low crop, head output size (== h, w when up == 1)
    // implicit-GEMM convolution (conv_k > 0): one M tile = a PH x PW patch of output pixels of one image;
    // K blocks run over taps x 64-channel blocks; A comes from a 4-D tensor map {C, W, H, B}
    int conv_k, conv_stride, conv_pad, conv_cblocks;
    int Hi, Wi, Ho, Wo, tiles_x, tiles_y;
    // residual add before the ReLU (torchvision BasicBlock / Bottleneck): res[m][res_col_off + n]
    const __nv_bfloat16* res; int ld_res; int res_col_off;
    // debug (SIMT) operand views
    const __nv_bfloat16* a; int lda; const __nv_bfloat16* wgt; int ldw;
    // per-image weights (implicit-GEMM conv only; squeeze-excitation projections): image b reads weight rows
    // [b * w_img_rows, (b + 1) * w_img_rows) of B; 0 = one weight matrix for the whole batch
    int w_img_rows;
};

constexpr int PH = 8, PW = 16;     // conv output patch per M tile (PH * PW == BM)

// tile row (== TMEM lane) -> output row index m, or -1 if outside the tensor
__device__ __forceinline__ int tile_row_to_m(const GemmArgs& g, int m_blk, int row) {
    if (g.conv_k == 0) {
        const int m = m_blk * BM + row;
        return m < g.M ? m : -1;
    }
    const int per_img = g.tiles_x * g.tiles_y;
    const int b = m_blk / per_img, t = m_blk - b * per_img;
    const int oy = (t / g.tiles_x) * PH + row / PW, ox = (t % g.tiles_x) * PW + row % PW;
    if (oy >= g.Ho || ox >= g.Wo) return -1;
    return (b * g.Ho + oy) * g.Wo + ox;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float softplus_f(float x) {   // torch softplus beta=1 threshold=20 (heads.py:378)
    return x > 20.0f ? x : log1pf(expf(x));
}
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }
// fused activation codes of the C ABI (include/pifpaf_b200.h): 0 none, 1 ReLU, 2 ReLU6, 3 Hardswish
// (torch.nn.Hardswish: x * min(max(x + 3, 0), 6) / 6, here with the reciprocal: within one ulp); applied in f32 before
// the bf16 rounding.  Codes 0..2 are one clamp whose bounds the compiler hoists out of the epilogue loops.
__device__ __forceinline__ float act_f(float x, int act) {
    if (act == 3) return x * fminf(fmaxf(x + 3.f, 0.f), 6.f) * (1.f / 6.f);
    return fminf(fmaxf(x, act ? 0.f : -INFINITY), act == 2 ? 6.f : INFINITY);
}

// Blackwell 256-bit global store (STG.E.256): p must be 32-byte aligned
__device__ __forceinline__ void st_global_256(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d,
                                              uint32_t e, uint32_t f, uint32_t g, uint32_t h) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "l"(p), "r"(a), "r"(b), "r"(c), "r"(d), "r"(e), "r"(f), "r"(g), "r"(h) : "memory");
}

// store `cnt` (<= 16) consecutive 32-bit words from registers to p (4-byte aligned, LEAD words before the
// first 16-byte boundary): scalar lead-in, 16-byte vectors, scalar tail.  Fully unrolled (no local memory).
template <int LEAD>
__device__ __forceinline__ void store_words(uint32_t* p, const uint32_t (&w)[CHUNK], int cnt) {
#pragma unroll
    for (int i = 0; i < LEAD; i++)
        if (i < cnt) p[i] = w[i];
#pragma unroll
    for (int i = LEAD; i + 4 <= CHUNK; i += 4) {
        if (i + 4 <= cnt) {
            *reinterpret_cast<uint4*>(p + i) = make_uint4(w[i], w[i + 1], w[i + 2], w[i + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (i + j < cnt) p[i + j] = w[i + j];
        }
    }
#pragma unroll
    for (int i = LEAD + (CHUNK - LEAD) / 4 * 4; i < CHUNK; i++)
        if (i < cnt) p[i] = w[i];
}

// Epilogue for one warp: 32 rows (lane == row) x CHUNK columns starting at GEMM column n0.
// acc[] holds this lane's CHUNK accumulators.  Every lane writes its own row with 16-byte vector stores
// (full 32-byte sectors), no shared-memory staging.
// bias: pointer to this chunk's CHUNK biases (shared memory in the tensor-core kernel, global in the debug
// kernel).  src_row: this lane's row of the pass-through tile at the chunk's first column (shared memory, filled
// by TMA) or nullptr to read it from global memory.
// dest: the MODE_SCATTER destination table (shared memory in the tensor-core kernel: a global load per chunk put
// 11 warps per issue on the long scoreboard, ncu round 1; global in the debug kernel)
// EXT: activation codes 2 / 3 (act_f) and per-image weights; the EXT = false instantiations are the ReLU-only kernels
// the ShuffleNetV2K / ResNet ops run (instruction for instruction the code they ran before activation codes existed)
template <bool EXT>
__device__ __forceinline__ void epilogue_chunk(const GemmArgs& g, int m, int n0, const float* acc,
                                               const float* bias, const __nv_bfloat16* src_row,
                                               const DestGroup* dest) {
    float bv[CHUNK];
    {
        const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
        for (int j = 0; j < CHUNK / 4; j++) {
            const float4 b4 = bp[j];
            bv[4 * j] = b4.x; bv[4 * j + 1] = b4.y; bv[4 * j + 2] = b4.z; bv[4 * j + 3] = b4.w;
        }
    }
    if (m < 0) return;
    if (g.mode == MODE_HEADS) {
        const int b = m / g.hw, pix = m - b * g.hw;
        const int y = pix / g.w, x = pix - y * g.w;
        const int out_hw = g.out_h * g.out_w;
#pragma unroll
        for (int j = 0; j < CHUNK; j++) {
            const int n = n0 + j;
            if (n >= g.N) break;
            const HeadCol hc = g.head_cols[n];
            // PixelShuffle(up) + crop [low, size - high) (heads.py:333-343): conv channel c*up*up + dy*up + dx of
            // cell (y, x) is output channel c at (y*up + dy - low, x*up + dx - low)
            const int oy = y * g.up + (hc.sub >> 8) - g.up_low, ox = x * g.up + (hc.sub & 255) - g.up_low;
            if (oy < 0 || oy >= g.out_h || ox < 0 || ox >= g.out_w) continue;
            float v = acc[j] + bv[j];
            if (hc.op == 1) v = sigmoid_f(v);
            else if (hc.op == 2) v += (float)ox;
            else if (hc.op == 3) v += (float)oy;
            else if (hc.op == 4) v = softplus_f(v);
            g.head_base[hc.head][((size_t)b * g.head_planes[hc.head] + hc.plane) * out_hw + oy * g.out_w + ox] = v;
        }
        return;
    }
    if (g.mode == MODE_SCATTER) {
        uint32_t w[CHUNK / 2];
#pragma unroll
        for (int j = 0; j < CHUNK; j += 2) {
            float a0 = acc[j] + bv[j], a1 = acc[j + 1] + bv[j + 1];
            if (g.relu) {
                if (EXT) { a0 = act_f(a0, g.relu); a1 = act_f(a1, g.relu); }
                else { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
            }
            w[j >> 1] = pack_bf16(a0, a1);
        }
        if (g.debug & 1) { if (w[0] == 0x12345u && w[5] == 0x54321u) g.dest[0].base[0] = __float2bfloat16(0.f); return; }
        if (n0 < g.N) {
            // debug 8 (timing only, wrong results): every piece goes to the first destination tensor, as one contiguous row
            DestGroup d = dest[n0 >> 4];
            if (g.debug & 8) { d = dest[0]; d.base += n0; }
            // debug 16 (timing only): every piece as its own [pixels][piece width] tensor (rows of one piece contiguous)
            if (g.debug & 16) { const int pw = d.pad >> 16, ci = d.pad & 0xffff; d.base = d.base - ci + (size_t)0; d.ld = pw; d.base += ci; }
            st_global_256(d.base + (size_t)m * d.ld, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7]);
        }
        return;
    }
    if (g.mode == MODE_PLAIN) {
        uint32_t w[CHUNK / 2];
        float rv[CHUNK];
        if (g.res != nullptr) {
            const uint4* rp = reinterpret_cast<const uint4*>(g.res + (size_t)m * g.ld_res + g.res_col_off + n0);
            const uint4 r0 = __ldg(rp), r1 = __ldg(rp + 1);
            const uint32_t rw[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
            for (int j = 0; j < 8; j++) {
                rv[2 * j] = __uint_as_float(rw[j] << 16);
                rv[2 * j + 1] = __uint_as_float(rw[j] & 0xffff0000u);
            }
        } else {
#pragma unroll
            for (int j = 0; j < CHUNK; j++) rv[j] = 0.f;
        }
#pragma unroll
        for (int j = 0; j < CHUNK; j += 2) {
            float a0 = acc[j] + bv[j] + rv[j], a1 = acc[j + 1] + bv[j + 1] + rv[j + 1];
            if (g.relu) {
                if (EXT) { a0 = act_f(a0, g.relu); a1 = act_f(a1, g.relu); }
                else { a0 = fmaxf(a0, 0.f); a1 = fmaxf(a1, 0.f); }
            }
            w[j >> 1] = pack_bf16(a0, a1);
        }
        if (g.debug & 1) { if (w[0] == 0x12345u && w[5] == 0x54321u) g.out[0] = __float2bfloat16(0.f); return; }
        // 16 bf16 = 32 bytes, 32-byte aligned (ldo % 16 == 0, out_col_off % 16 == 0, n0 % 16 == 0)
        uint4* dst = reinterpret_cast<uint4*>(g.out + (size_t)m * g.ldo + g.out_col_off + n0);
        const int n_pad8 = (g.N + 7) & ~7;
        if (n0 + 8 < n_pad8) {
            st_global_256(dst, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7]);
        } else if (n0 < n_pad8) {
            dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
        }
        return;
    }
    // MODE_SHUFFLE: word n = { src0[m][n] (logical channel 2n), conv[m][n] (logical 2n+1) }
    const uint4* sp = src_row != nullptr
        ? reinterpret_cast<const uint4*>(src_row)
        : reinterpret_cast<const uint4*>(g.src0 + (size_t)m * g.ld0 + g.src0_col_off + n0);
    const uint4 s0 = sp[0], s1 = sp[1];
    const uint32_t sw[8] = {s0.x, s0.y, s0.z, s0.w, s1.x, s1.y, s1.z, s1.w};
    uint32_t w[CHUNK];
#pragma unroll
    for (int j = 0; j < CHUNK; j++) {
        float a = acc[j] + bv[j];
        if (g.relu) a = EXT ? act_f(a, g.relu) : fmaxf(a, 0.f);
        const uint32_t src_bits = (j & 1) ? (sw[j >> 1] >> 16) : (sw[j >> 1] & 0xffffu);
        const __nv_bfloat16 hb = __float2bfloat16_rn(a);
        w[j] = src_bits | (static_cast<uint32_t>(__bfloat16_as_ushort(hb)) << 16);
    }
    // logical channel 2n, 2n+1 == physical word n (gap-free layout): 64 bytes per lane, 64-byte aligned
    uint32_t* row = reinterpret_cast<uint32_t*>(g.out) + (size_t)m * (g.ldo >> 1) + (g.out_col_off >> 1) + n0;
    const int cnt = min(CHUNK, g.N - n0);
    if (cnt == CHUNK) {
        st_global_256(row, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7]);
        st_global_256(row + 8, w[8], w[9], w[10], w[11], w[12], w[13], w[14], w[15]);
    } else {
        store_words<0>(row, w, cnt);
    }
}

// ------------------------------------------------------------------ tcgen05 GEMM
template <bool EXT>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
k_gemm_tc(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
          const __grid_constant__ CUtensorMap tmap_src, GemmArgs g) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // carve: [stages][A 16 KB | B block_n*128 B] then barriers, tmem ptr, staging
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int a_bytes = BM * BK * 2;
    const int b_bytes = g.block_n * BK * 2;
    // weights-resident mode: the ring carries only A; the CTA's weight tile (all K blocks of ONE n block) is
    // loaded once -- weights are otherwise re-fetched from L2 for every M tile and outweigh the A traffic
    const int stage_bytes = a_bytes + (g.b_resident ? 0 : b_bytes);
    unsigned char* b_res = smem + (size_t)g.stages * stage_bytes;
    const size_t b_res_bytes = g.b_resident ? (size_t)g.num_k_blocks * b_bytes : 0;
    // pass-through tiles of the fused shuffle: [2 accumulator stages][BM rows][block_n] bf16, filled by TMA
    const int src_bytes = g.src_tma ? BM * g.block_n * 2 : 0;
    unsigned char* src_tiles = b_res + b_res_bytes;
    float* bias_s = reinterpret_cast<float*>(src_tiles + 2 * (size_t)src_bytes);   // [n_blocks * block_n]
    DestGroup* dest_s = reinterpret_cast<DestGroup*>(bias_s + g.n_blocks * g.block_n);   // [n_blocks * block_n / 16]
    unsigned char* tail = reinterpret_cast<unsigned char*>(dest_s + g.n_blocks * g.block_n / CHUNK);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);            // [stages]
    uint64_t* empty_bar = full_bar + g.stages;                          // [stages]
    uint64_t* tmem_full = empty_bar + g.stages;                         // [2]
    uint64_t* tmem_empty = tmem_full + 2;                               // [2]
    uint64_t* src_full = tmem_empty + 2;                                // [2]
    uint64_t* b_full = src_full + 2;                                    // [1]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t tmem_cols = (2 * g.block_n <= 32) ? 32 : (2 * g.block_n <= 64) ? 64 : (2 * g.block_n <= 128) ? 128
                               : (2 * g.block_n <= 256) ? 256 : 512;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmap_a);
        tma_prefetch_desc(&tmap_b);
        if (g.src_tma || g.mc) tma_prefetch_desc(&tmap_src);
    }
    for (int i = threadIdx.x; i < g.n_blocks * g.block_n; i += GEMM_THREADS) bias_s[i] = g.bias[i];
    if (g.mode == MODE_SCATTER)
        for (int i = threadIdx.x; i < g.n_blocks * g.block_n / CHUNK; i += GEMM_THREADS) dest_s[i] = g.dest[i];
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < g.stages; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], g.mc ? 2 : 1); }
            for (int a = 0; a < 2; a++) {
                mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], EPI_WARPS); mbar_init(&src_full[a], 1);
            }
            mbar_init(b_full, 1);
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(tmem_ptr, tmem_cols);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // the peer's barriers must be initialised before anything of this CTA (multicast data, commit arrivals) reaches them
    if (g.mc) cluster_sync_all();
    const uint32_t mc_rank = g.mc ? cluster_ctarank() : 0;
    // the resident weight tile does not depend on the predecessor kernel: its loads go out before the grid-dependency
    // wait and land while the predecessor's last CTAs drain (counts at 8 images per GPU, where a launch lasts 15-40 us)
    if (warp == 0 && lane == 0 && g.b_resident) {
        mbar_expect_tx(b_full, (uint32_t)b_res_bytes);
        for (int kb = 0; kb < g.num_k_blocks; kb++)
            tma_load_2d(b_res + (size_t)kb * b_bytes, &tmap_b, b_full, kb * BK, (int)(blockIdx.x % g.n_blocks) * g.block_n);
    }
    // (after the TMEM allocation: a dependent CTA that becomes co-resident must not take the columns first)
    pdl_launch_dependents();
    pdl_wait();

    // tile schedule: streaming mode walks (m_blk, n_blk) tiles round-robin over the CTAs; weights-resident mode
    // pins one n block per CTA (gridDim.x is a multiple of n_blocks) and walks M tiles only
    const int num_tiles = g.b_resident ? 0 : g.m_blocks * g.n_blocks;
    const int my_n = g.b_resident ? (int)(blockIdx.x % g.n_blocks) : 0;
    const int m_first = g.b_resident ? (int)(blockIdx.x / g.n_blocks) : 0;
    const int m_step = g.b_resident ? (int)(gridDim.x / g.n_blocks) : 0;
#define PIFPAF_TILE_LOOP(m_blk, n_blk)                                                                             \
    for (int it__ = g.b_resident ? m_first : (int)blockIdx.x, m_blk = 0, n_blk = 0;                                 \
         (g.b_resident ? it__ < g.m_blocks : it__ < num_tiles) &&                                                   \
         ((m_blk = g.b_resident ? it__ : it__ / g.n_blocks), (n_blk = g.b_resident ? my_n : it__ % g.n_blocks), true); \
         it__ += g.b_resident ? m_step : (int)gridDim.x)

    if (warp == 0) {
        // ===== TMA producer (one elected lane) =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int sacc = 0; uint32_t sacc_phase = 0;
            PIFPAF_TILE_LOOP(m_blk, n_blk) {
                int cb = 0, cy = 0, cx = 0, cimg = 0;
                if (g.conv_k > 0) {
                    const int per_img = g.tiles_x * g.tiles_y;
                    cimg = m_blk / per_img;
                    const int t = m_blk - cimg * per_img;
                    cy = (t / g.tiles_x) * PH * g.conv_stride - g.conv_pad;
                    cx = (t % g.tiles_x) * PW * g.conv_stride - g.conv_pad;
                }
                for (int kb = 0; kb < g.num_k_blocks; kb++) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char* sa = smem + (size_t)stage * stage_bytes;
                    unsigned char* sb = sa + a_bytes;
                    mbar_expect_tx(&full_bar[stage], (uint32_t)stage_bytes);
                    if (g.conv_k > 0) {
                        const int tap = kb / g.conv_cblocks;
                        cb = kb - tap * g.conv_cblocks;
                        tma_load_4d(sa, &tmap_a, &full_bar[stage], cb * BK, cx + tap % g.conv_k, cy + tap / g.conv_k, cimg);
                    } else if (g.mc) {
                        // this CTA's half of the stage (64 rows = 8 KB, a whole number of swizzle atoms) to both CTAs; the
                        // peer sends the other half.  The 16 KB expected above arrive from the two loads.
                        tma_load_2d_mc(sa + mc_rank * (BM / 2) * BK * 2, &tmap_src, &full_bar[stage], g.a_col0 + kb * BK,
                                       m_blk * BM + (int)mc_rank * (BM / 2), (uint16_t)3);
                    } else {
                        tma_load_2d(sa, &tmap_a, &full_bar[stage], g.a_col0 + kb * BK, m_blk * BM);
                    }
                    if (!g.b_resident) tma_load_2d(sb, &tmap_b, &full_bar[stage], kb * BK, n_blk * g.block_n + (EXT ? cimg * g.w_img_rows : 0));
                    if (++stage == g.stages) { stage = 0; phase ^= 1; }
                }
                if (g.src_tma) {
                    // pass-through tile of this output tile; its buffer is free once the epilogue that used this
                    // accumulator stage two tiles ago has released it
                    mbar_wait(&tmem_empty[sacc], sacc_phase ^ 1);
                    mbar_expect_tx(&src_full[sacc], (uint32_t)src_bytes);
                    tma_load_2d(src_tiles + (size_t)sacc * src_bytes, &tmap_src, &src_full[sacc],
                                n_blk * g.block_n, m_blk * BM);
                    if (++sacc == 2) { sacc = 0; sacc_phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            const uint32_t idesc = make_instr_desc(BM, g.block_n);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            if (g.b_resident) mbar_wait(b_full, 0);
            PIFPAF_TILE_LOOP(m_blk, n_blk) {
                (void)m_blk; (void)n_blk;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * g.block_n);
                for (int kb = 0; kb < g.num_k_blocks; kb++) {
                    mbar_wait(&full_bar[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint32_t sb = g.b_resident ? smem_u32(b_res + (size_t)kb * b_bytes) : sa + a_bytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adesc = make_smem_desc(sa + k * UMMA_K * 2);
                        const uint64_t bdesc = make_smem_desc(sb + k * UMMA_K * 2);
                        if (!(g.debug & 2)) umma_bf16(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    // frees the smem slot when the MMAs retire (multicast mode: in both CTAs, each refills half of it)
                    if (g.mc) umma_commit_mc(&empty_bar[stage], (uint16_t)3); else umma_commit(&empty_bar[stage]);
                    if (++stage == g.stages) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full[acc]);                // accumulator ready for the epilogue
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue warps: TMEM lane quadrant = warp % 4; the EPI_WARPS/4 warps of a quadrant split the
        // column chunks evenly =====
        const int q = warp & 3;
        const int n_chunks = g.block_n / CHUNK;
        const int part = (warp - 2) >> 2, parts = EPI_WARPS / 4;
        const int c_begin = n_chunks * part / parts;
        const int c_end = n_chunks * (part + 1) / parts;
        int acc = 0; uint32_t acc_phase = 0;
        PIFPAF_TILE_LOOP(m_blk, n_blk) {
            mbar_wait(&tmem_full[acc], acc_phase);
            tcgen05_fence_after();
            if (g.src_tma) mbar_wait(&src_full[acc], acc_phase);
            const int m = tile_row_to_m(g, m_blk, q * 32 + lane);
            const __nv_bfloat16* src_tile_row = reinterpret_cast<const __nv_bfloat16*>(
                src_tiles + (size_t)acc * src_bytes) + (size_t)(q * 32 + lane) * g.block_n;
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (uint32_t)(acc * g.block_n);
            // software-pipelined TMEM reads: the load of chunk ci+1 is in flight while chunk ci is processed
            uint32_t va[CHUNK], vb[CHUNK];
            auto process = [&](int ci, const uint32_t* v) {
                const int c = ci * CHUNK;
                float accf[CHUNK];
#pragma unroll
                for (int j = 0; j < CHUNK; j++) accf[j] = __uint_as_float(v[j]);
                const int n0 = n_blk * g.block_n + c;
                if (n0 < ((g.N + 7) & ~7))
                    epilogue_chunk<EXT>(g, m, n0, accf, bias_s + n0, g.src_tma ? src_tile_row + c : nullptr, dest_s);
            };
            if (g.debug & 4) {                       // timing experiment: release the accumulator without reading it
                for (int ci = c_begin; ci < c_end; ci++) {
#pragma unroll
                    for (int j = 0; j < CHUNK; j++) va[j] = (uint32_t)(ci + j + m);
                    process(ci, va);
                }
                tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tmem_empty[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                continue;
            }
            if (c_begin < c_end) tmem_ld16_async(t_row + (uint32_t)(c_begin * CHUNK), va);
            for (int ci = c_begin; ci < c_end; ci += 2) {
                tmem_ld_wait(va);
                if (ci + 1 < c_end) tmem_ld16_async(t_row + (uint32_t)((ci + 1) * CHUNK), vb);
                process(ci, va);
                if (ci + 1 < c_end) {
                    tmem_ld_wait(vb);
                    if (ci + 2 < c_end) tmem_ld16_async(t_row + (uint32_t)((ci + 2) * CHUNK), va);
                    process(ci + 1, vb);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    // no CTA of a multicast pair may exit while the other can still send data or barrier arrivals into it
    if (g.mc) cluster_sync_all();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

// ------------------------------------------------------------------ tcgen05 GEMM, CTA pairs (cta_group::2)
// Measured (profiles/r2_history.md, sessions l-n): the weights-resident GEMMs of stage 3 are bound by the bytes of A
// in flight -- the resident weight tile (135-160 KB) leaves 4-5 stages of 16 KB, a load takes 1.7 us under load, and a
// stage is only free once its MMAs have retired, so loads, MMAs and stores ADD (0.091 + 0.03 + 0.03 ms) instead of
// overlapping; the streaming GEMMs of stage 4 / conv5 run into the L2 -> SM cap (12 TB/s) re-reading the weights.
// Both get relief from the two-SM MMA: the two CTAs of a cluster compute ONE 256 x block_n tile; each CTA stages its
// own 128 rows of A and only HALF of the weight tile (rows [rank * block_n / 2, +block_n / 2) of the n block), the
// leader issues tcgen05.mma.cta_group::2 (M = 256) and each CTA's TMEM receives the accumulator rows of its own A
// half.  Per SM: half the weight bytes in shared memory (twice the A stages) and half the weight traffic from L2.
//   full[stage]    (leader only)  both CTAs' TMA loads complete bytes there (cta_group::2 loads with the peer bit
//                                 of the barrier address cleared); the leader's producer arms it with the pair's total
//   empty[stage]   (each CTA)     tcgen05.commit.cta_group::2 ... multicast to both CTAs when the MMAs have read it
//   tmem_full[a]   (each CTA)     the same commit, after the last K block of a tile
//   tmem_empty[a]  (leader only)  the 2 x 16 epilogue warps of the pair arrive there (remote arrive from the peer)
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;      // shared::cluster address of the same offset in the even CTA of the pair
constexpr int PAIR_MAX_STAGES = 12;

__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & PEER_BIT_MASK) : "memory");
}

template <bool EXT>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
k_gemm_tc2(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_bh, GemmArgs g) {
    extern __shared__ __align__(1024) unsigned char smem_raw2[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw2) + 1023) & ~uintptr_t(1023));
    const int half_n = g.block_n / 2;
    const int a_bytes = BM * BK * 2;
    const int bh_bytes = half_n * BK * 2;                       // this CTA's half of one K block of the weight tile
    const int stage_bytes = a_bytes + (g.b_resident ? 0 : bh_bytes);
    unsigned char* b_res = smem + (size_t)g.pair_stages * stage_bytes;
    const size_t b_res_bytes = g.b_resident ? (size_t)g.num_k_blocks * bh_bytes : 0;
    float* bias_s = reinterpret_cast<float*>(b_res + ((b_res_bytes + 1023) & ~(size_t)1023));
    DestGroup* dest_s = reinterpret_cast<DestGroup*>(bias_s + g.n_blocks * g.block_n);
    unsigned char* tail = reinterpret_cast<unsigned char*>(dest_s + g.n_blocks * g.block_n / CHUNK);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);            // [stages]   used in the leader
    uint64_t* empty_bar = full_bar + g.pair_stages;                     // [stages]
    uint64_t* tmem_full = empty_bar + g.pair_stages;                    // [2]
    uint64_t* tmem_empty = tmem_full + 2;                               // [2]        used in the leader
    uint64_t* b_full = tmem_empty + 2;                                  // [1]        used in the leader
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const uint32_t tmem_cols = (2 * g.block_n <= 32) ? 32 : (2 * g.block_n <= 64) ? 64 : (2 * g.block_n <= 128) ? 128
                               : (2 * g.block_n <= 256) ? 256 : 512;

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_a); tma_prefetch_desc(&tmap_bh); }
    for (int i = threadIdx.x; i < g.n_blocks * g.block_n; i += GEMM_THREADS) bias_s[i] = g.bias[i];
    if (g.mode == MODE_SCATTER)
        for (int i = threadIdx.x; i < g.n_blocks * g.block_n / CHUNK; i += GEMM_THREADS) dest_s[i] = g.dest[i];
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < g.pair_stages; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
            for (int a = 0; a < 2; a++) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 2 * EPI_WARPS); }
            mbar_init(b_full, 1);
            fence_barrier_init();
        }
        __syncwarp();
        // the same warp of both CTAs: one allocation, the same columns in both tensor memories
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_ptr)), "r"(tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                 // the peer's barriers exist before any load / commit / arrive reaches them
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // resident weights: loaded before the grid-dependency wait (they do not depend on the predecessor kernel)
    if (warp == 0 && lane == 0 && g.b_resident) {
        const int my_n0 = (int)(blockIdx.x >> 1) % g.n_blocks;
        if (rank == 0) mbar_expect_tx(b_full, (uint32_t)(2 * b_res_bytes));
        const uint32_t lb = smem_u32(b_full) & PEER_BIT_MASK;
        for (int kb = 0; kb < g.num_k_blocks; kb++)
            tma_load_2d_pair(b_res + (size_t)kb * bh_bytes, &tmap_bh, lb, kb * BK, my_n0 * g.block_n + (int)rank * half_n);
    }
    pdl_launch_dependents();
    pdl_wait();

    // tile schedule over PAIRS (cluster index): weights-resident mode pins one n block per pair and walks the
    // 256-row tiles; streaming mode walks (m256, n_blk) tiles round-robin
    const int pair = (int)(blockIdx.x >> 1), n_pairs = (int)(gridDim.x >> 1);
    const int m2_blocks = (g.M + 2 * BM - 1) / (2 * BM);
    const int num_tiles = g.b_resident ? 0 : m2_blocks * g.n_blocks;
    const int my_n = g.b_resident ? pair % g.n_blocks : 0;
    const int m_first = g.b_resident ? pair / g.n_blocks : 0;
    const int m_step = g.b_resident ? n_pairs / g.n_blocks : 0;
#define PIFPAF_PAIR_LOOP(m_blk, n_blk)                                                                             \
    for (int it__ = g.b_resident ? m_first : pair, m_blk = 0, n_blk = 0;                                            \
         (g.b_resident ? it__ < m2_blocks : it__ < num_tiles) &&                                                    \
         ((m_blk = g.b_resident ? it__ : it__ / g.n_blocks), (n_blk = g.b_resident ? my_n : it__ % g.n_blocks), true); \
         it__ += g.b_resident ? m_step : n_pairs)

    if (warp == 0) {
        // ===== TMA producer (one lane in each CTA) =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            PIFPAF_PAIR_LOOP(m_blk, n_blk) {
                for (int kb = 0; kb < g.num_k_blocks; kb++) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    unsigned char* sa = smem + (size_t)stage * stage_bytes;
                    if (rank == 0) mbar_expect_tx(&full_bar[stage], (uint32_t)(2 * stage_bytes));
                    const uint32_t lb = smem_u32(&full_bar[stage]) & PEER_BIT_MASK;
                    tma_load_2d_pair(sa, &tmap_a, lb, g.a_col0 + kb * BK, m_blk * 2 * BM + (int)rank * BM);
                    if (!g.b_resident)
                        tma_load_2d_pair(sa + a_bytes, &tmap_bh, lb, kb * BK, n_blk * g.block_n + (int)rank * half_n);
                    if (++stage == g.pair_stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one lane of the LEADER CTA =====
        if (lane == 0 && rank == 0) {
            const uint32_t idesc = make_instr_desc(2 * BM, g.block_n);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            if (g.b_resident) mbar_wait(b_full, 0);
            PIFPAF_PAIR_LOOP(m_blk, n_blk) {
                (void)m_blk; (void)n_blk;
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * g.block_n);
                for (int kb = 0; kb < g.num_k_blocks; kb++) {
                    mbar_wait(&full_bar[stage], phase);
                    tcgen05_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)stage * stage_bytes);
                    const uint32_t sb = g.b_resident ? smem_u32(b_res + (size_t)kb * bh_bytes) : sa + a_bytes;
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adesc = make_smem_desc(sa + k * UMMA_K * 2);
                        const uint64_t bdesc = make_smem_desc(sb + k * UMMA_K * 2);
                        umma_bf16_pair(d_tmem, adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                    }
                    umma_commit_pair(&empty_bar[stage]);
                    if (++stage == g.pair_stages) { stage = 0; phase ^= 1; }
                }
                umma_commit_pair(&tmem_full[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue warps of both CTAs: this CTA's 128 rows of the tile =====
        const int q = warp & 3;
        const int n_chunks = g.block_n / CHUNK;
        const int part = (warp - 2) >> 2, parts = EPI_WARPS / 4;
        const int c_begin = n_chunks * part / parts;
        const int c_end = n_chunks * (part + 1) / parts;
        int acc = 0; uint32_t acc_phase = 0;
        PIFPAF_PAIR_LOOP(m_blk, n_blk) {
            mbar_wait(&tmem_full[acc], acc_phase);
            tcgen05_fence_after();
            const int mrow = m_blk * 2 * BM + (int)rank * BM + q * 32 + lane;
            const int m = mrow < g.M ? mrow : -1;
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (uint32_t)(acc * g.block_n);
            uint32_t va[CHUNK], vb[CHUNK];
            auto process = [&](int ci, const uint32_t* v) {
                const int c = ci * CHUNK;
                float accf[CHUNK];
#pragma unroll
                for (int j = 0; j < CHUNK; j++) accf[j] = __uint_as_float(v[j]);
                const int n0 = n_blk * g.block_n + c;
                if (n0 < ((g.N + 7) & ~7)) epilogue_chunk<EXT>(g, m, n0, accf, bias_s + n0, nullptr, dest_s);
            };
            if (c_begin < c_end) tmem_ld16_async(t_row + (uint32_t)(c_begin * CHUNK), va);
            for (int ci = c_begin; ci < c_end; ci += 2) {
                tmem_ld_wait(va);
                if (ci + 1 < c_end) tmem_ld16_async(t_row + (uint32_t)((ci + 1) * CHUNK), vb);
                process(ci, va);
                if (ci + 1 < c_end) {
                    tmem_ld_wait(vb);
                    if (ci + 2 < c_end) tmem_ld16_async(t_row + (uint32_t)((ci + 2) * CHUNK), va);
                    process(ci + 1, vb);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_leader(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    cluster_sync_all();                 // nobody leaves (or frees tensor memory) while the pair is still at work
    if (warp == 1) {
        tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

// ------------------------------------------------------------------ SIMT debug GEMM (tests only)
// One warp per 32 rows x CHUNK columns; same epilogue as the tensor-core kernel.
__global__ void __launch_bounds__(128) k_gemm_simt(GemmArgs g) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_chunks = g.n_blocks * g.block_n / CHUNK;
    const long long total = (long long)g.m_blocks * 4 * n_chunks;        // 4 row quarters per M tile
    for (long long job = (long long)blockIdx.x * 4 + warp; job < total; job += (long long)gridDim.x * 4) {
        const int ch = (int)(job % n_chunks);
        const int mq = (int)(job / n_chunks);
        const int m_blk = mq >> 2, row = (mq & 3) * 32 + lane;
        const int n0 = ch * CHUNK;
        const int m = tile_row_to_m(g, m_blk, row);
        float acc[CHUNK];
#pragma unroll
        for (int j = 0; j < CHUNK; j++) acc[j] = 0.f;
        if (m >= 0) {
            if (g.conv_k == 0) {
                for (int k = 0; k < g.K; k++) {
                    const float a = __bfloat162float(g.a[(size_t)m * g.lda + k]);
#pragma unroll
                    for (int j = 0; j < CHUNK; j++) {
                        const int n = n0 + j;
                        const float wv = (n < g.N) ? __bfloat162float(g.wgt[(size_t)n * g.ldw + k]) : 0.f;
                        acc[j] = fmaf(a, wv, acc[j]);
                    }
                }
            } else {
                const int ox = m % g.Wo, oy = (m / g.Wo) % g.Ho, b = m / (g.Wo * g.Ho);
                for (int tap = 0; tap < g.conv_k * g.conv_k; tap++) {
                    const int iy = oy * g.conv_stride - g.conv_pad + tap / g.conv_k;
                    const int ix = ox * g.conv_stride - g.conv_pad + tap % g.conv_k;
                    if (iy < 0 || iy >= g.Hi || ix < 0 || ix >= g.Wi) continue;
                    const __nv_bfloat16* ap = g.a + ((size_t)(b * g.Hi + iy) * g.Wi + ix) * g.lda;
                    for (int k = 0; k < g.K; k++) {
                        const float a = __bfloat162float(ap[k]);
#pragma unroll
                        for (int j = 0; j < CHUNK; j++) {
                            const int n = n0 + j;
                            const float wv = (n < g.N)
                                ? __bfloat162float(g.wgt[((size_t)b * g.w_img_rows + n) * g.ldw + (size_t)tap * g.conv_cblocks * BK + k]) : 0.f;
                            acc[j] = fmaf(a, wv, acc[j]);
                        }
                    }
                }
            }
        }
        if (n0 < ((g.N + 7) & ~7)) epilogue_chunk<true>(g, m, n0, acc, g.bias + n0, nullptr, g.dest);
    }
}

// ------------------------------------------------------------------ depthwise kxk conv, NHWC bf16
// one thread: one output pixel x 8 channels (16-byte vectors); weights [k*k][C8*8] f32, bias [C]
struct DwArgs {
    const __nv_bfloat16* in; int ld_in; int in_col_off;
    __nv_bfloat16* out; int ld_out; int out_col_off;
    const float* weight; const float* bias;
    int B, Hin, Win, Hout, Wout, C8, kernel, stride, pad, relu;
};

// bf16x2 word -> two floats (bf16 -> f32 is a 16-bit shift)
__device__ __forceinline__ void unpack8(const uint4& v, float* f) {
    f[0] = __uint_as_float(v.x << 16); f[1] = __uint_as_float(v.x & 0xffff0000u);
    f[2] = __uint_as_float(v.y << 16); f[3] = __uint_as_float(v.y & 0xffff0000u);
    f[4] = __uint_as_float(v.z << 16); f[5] = __uint_as_float(v.z & 0xffff0000u);
    f[6] = __uint_as_float(v.w << 16); f[7] = __uint_as_float(v.w & 0xffff0000u);
}

// Register-tiled depthwise 5x5: one thread = 8 channels x DW_OX consecutive output pixels of one row.
// Each input vector is loaded once and feeds every output/tap it touches; the 5x8 weights of a kernel row
// stay in registers.  f32 accumulate.  (k == 5 only; other kernels take the generic path below.)
constexpr int DW_OX = 4;
constexpr int DW_OY = 8;

template <int S>
__global__ void __launch_bounds__(256) k_dwconv5(DwArgs a) {
    constexpr int NCOL = (DW_OX - 1) * S + 5;
    const int strips = (a.Wout + DW_OX - 1) / DW_OX;
    const int ytiles = (a.Hout + DW_OY - 1) / DW_OY;
    const long long total = (long long)a.B * ytiles * strips * DW_OY * a.C8;
    const int C = a.C8 * 8;
    // thread order: channels fastest (coalesced 16-byte vectors), then DW_OY vertically adjacent rows of the
    // same strip (their 5-row input windows overlap -> L1 hits), then strips, row tiles, images
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int c8 = (int)(t % a.C8);
        long long p = t / a.C8;
        const int yl = (int)(p % DW_OY); p /= DW_OY;
        const int sx = (int)(p % strips); p /= strips;
        const int oy = (int)(p % ytiles) * DW_OY + yl;
        const int b = (int)(p / ytiles);
        if (oy >= a.Hout) continue;
        const int ox0 = sx * DW_OX;
        const int ix0 = ox0 * S - a.pad;
        float acc[DW_OX][8];
        {
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(a.bias + c8 * 8));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(a.bias + c8 * 8 + 4));
#pragma unroll
            for (int o = 0; o < DW_OX; o++) {
                acc[o][0] = b0.x; acc[o][1] = b0.y; acc[o][2] = b0.z; acc[o][3] = b0.w;
                acc[o][4] = b1.x; acc[o][5] = b1.y; acc[o][6] = b1.z; acc[o][7] = b1.w;
            }
        }
#pragma unroll
        for (int ky = 0; ky < 5; ky++) {
            const int iy = oy * S - a.pad + ky;
            if (iy < 0 || iy >= a.Hin) continue;
            float w[5][8];
#pragma unroll
            for (int kx = 0; kx < 5; kx++) {
                const float* wp = a.weight + (size_t)(ky * 5 + kx) * C + c8 * 8;
                const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
                const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
                w[kx][0] = w0.x; w[kx][1] = w0.y; w[kx][2] = w0.z; w[kx][3] = w0.w;
                w[kx][4] = w1.x; w[kx][5] = w1.y; w[kx][6] = w1.z; w[kx][7] = w1.w;
            }
            const __nv_bfloat16* rowp = a.in + ((size_t)(b * a.Hin + iy) * a.Win) * a.ld_in + a.in_col_off + c8 * 8;
#pragma unroll
            for (int col = 0; col < NCOL; col++) {
                const int ix = ix0 + col;
                if (ix < 0 || ix >= a.Win) continue;
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(rowp + (size_t)ix * a.ld_in));
                float f[8];
                unpack8(v, f);
#pragma unroll
                for (int o = 0; o < DW_OX; o++) {
                    const int kx = col - o * S;       // compile-time after unrolling
                    if (kx < 0 || kx >= 5) continue;
#pragma unroll
                    for (int j = 0; j < 8; j++) acc[o][j] = fmaf(f[j], w[kx][j], acc[o][j]);
                }
            }
        }
#pragma unroll
        for (int o = 0; o < DW_OX; o++) {
            const int ox = ox0 + o;
            if (ox >= a.Wout) continue;
            if (a.relu) {
#pragma unroll
                for (int j = 0; j < 8; j++) acc[o][j] = fmaxf(acc[o][j], 0.f);
            }
            uint4 ov;
            ov.x = pack_bf16(acc[o][0], acc[o][1]); ov.y = pack_bf16(acc[o][2], acc[o][3]);
            ov.z = pack_bf16(acc[o][4], acc[o][5]); ov.w = pack_bf16(acc[o][6], acc[o][7]);
            *reinterpret_cast<uint4*>(a.out + ((size_t)(b * a.Hout + oy) * a.Wout + ox) * a.ld_out + a.out_col_off + c8 * 8) = ov;
        }
    }
}

// Depthwise 5x5 with TMA-staged input tiles.  A persistent CTA walks (channel block, image, tile) work items; the
// input window of an item ((TH-1)*S+5 x (TW-1)*S+5 pixels x 64 channels, 4-D tensor map, out-of-bounds zero fill
// == the conv padding) is streamed by TMA into an NSTAGE-deep shared-memory ring.  There is no CTA-wide barrier in
// the steady state: every warp counts itself out of a ring slot with one shared-memory atomic, and the warp that
// finishes a slot LAST re-arms it with the TMA of the item NSTAGE rounds ahead, so fast warps (edge tiles with
// out-of-range blocks) run ahead of slow ones by up to NSTAGE-1 items.
// Compute mapping (register blocking in BOTH spatial directions): one warp = one 4 x BW block of output pixels,
// one lane = one channel pair.  The lane keeps its 25x2 weights and a 4 x BW x 2 f32 accumulator in registers and
// reads every input pixel of the block's window exactly once (4 bytes per lane, 128 bytes per warp request: one
// conflict-free wavefront).
template <int S, int TH, int TW, int BW, int NSTAGE>
struct DwTile {
    static constexpr int IH = (TH - 1) * S + 5, IW = (TW - 1) * S + 5;
    static constexpr int BYTES = IH * IW * 64 * 2;
    static constexpr int WARPS = (TH / 4) * (TW / BW);
    static constexpr int THREADS = WARPS * 32;
    static constexpr int WIN_Y = 3 * S + 5;            // input window of a 4 x BW output block
    static constexpr int WIN_X = (BW - 1) * S + 5;
    static constexpr int SMEM = NSTAGE * BYTES + 128;
};

// position of a work item and its increment per persistent-loop step, kept as mixed-radix digits
// (channel block, image, tile row, tile column) so that the loop needs no integer division
struct DwPos { int c, b, y, x; };

__device__ __forceinline__ DwPos dw_decompose(int w, int per_c, int tiles_y, int tiles_x) {
    DwPos p;
    p.c = w / per_c; int r = w - p.c * per_c;
    p.b = r / (tiles_y * tiles_x); r -= p.b * tiles_y * tiles_x;
    p.y = r / tiles_x; p.x = r - p.y * tiles_x;
    return p;
}

__device__ __forceinline__ void dw_advance(DwPos& p, const DwPos& d, int B, int tiles_y, int tiles_x) {
    p.x += d.x; int carry = p.x >= tiles_x; p.x -= carry ? tiles_x : 0;
    p.y += d.y + carry; carry = p.y >= tiles_y; p.y -= carry ? tiles_y : 0;
    p.b += d.b + carry; carry = p.b >= B; p.b -= carry ? B : 0;
    p.c += d.c + carry;
}

// channel-block-FASTEST item order (CBF): item = (image, tile row, tile column, channel block) with the channel block
// as the fastest digit, so the 128-byte channel blocks of one pixel (352 / 704-byte pixels: most blocks straddle a
// 64-byte DRAM atom) and the halos of neighbouring tiles are fetched by CTAs running at the same time and meet in L2.
__device__ __forceinline__ DwPos dw_decompose_cf(int w, int cblks, int tiles_y, int tiles_x) {
    DwPos p;
    p.c = w % cblks; int r = w / cblks;
    p.x = r % tiles_x; r /= tiles_x;
    p.y = r % tiles_y; p.b = r / tiles_y;
    return p;
}

__device__ __forceinline__ void dw_advance_cf(DwPos& p, const DwPos& d, int cblks, int tiles_y, int tiles_x) {
    p.c += d.c; int carry = p.c >= cblks; p.c -= carry ? cblks : 0;
    p.x += d.x + carry; carry = p.x >= tiles_x; p.x -= carry ? tiles_x : 0;
    p.y += d.y + carry; carry = p.y >= tiles_y; p.y -= carry ? tiles_y : 0;
    p.b += d.b + carry;
}

template <int S, int TH, int TW, int BW, int NSTAGE, bool CBF = false>
__global__ void __launch_bounds__(DwTile<S, TH, TW, BW, NSTAGE>::THREADS, 2)
k_dwconv5_tma(const __grid_constant__ CUtensorMap tmap_in, DwArgs a) {
    using T = DwTile<S, TH, TW, BW, NSTAGE>;
    extern __shared__ __align__(128) unsigned char dsm_raw[];
    // align inside the shared window with pointer arithmetic on the array itself (keeps the address space known to
    // the compiler: LDS instead of generic loads)
    unsigned char* dsm = dsm_raw + ((128u - (smem_u32(dsm_raw) & 127u)) & 127u);
    __shared__ uint64_t full[NSTAGE];
    __shared__ int done[NSTAGE];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tiles_x = (a.Wout + TW - 1) / TW, tiles_y = (a.Hout + TH - 1) / TH;
    const int cblks = (a.C8 + 7) / 8;
    const int per_c = a.B * tiles_y * tiles_x;
    const int total = per_c * cblks;
    const int C = a.C8 * 8;
    // CBF: the channel block changes with (almost) every item, so the weights [25][C] + bias [C] are staged in
    // shared memory once per CTA and re-read from there (26 LDS.64 per item)
    const float* s_w = reinterpret_cast<const float*>(dsm + (size_t)NSTAGE * T::BYTES);
    if (CBF) {
        float* sw = reinterpret_cast<float*>(dsm + (size_t)NSTAGE * T::BYTES);
        for (int i = tid; i < 25 * C; i += T::THREADS) sw[i] = a.weight[i];
        for (int i = tid; i < C; i += T::THREADS) sw[25 * C + i] = a.bias[i];
    }
    auto decompose = [&](int w) { return CBF ? dw_decompose_cf(w, cblks, tiles_y, tiles_x) : dw_decompose(w, per_c, tiles_y, tiles_x); };
    auto advance = [&](DwPos& p, const DwPos& d) {
        if (CBF) dw_advance_cf(p, d, cblks, tiles_y, tiles_x); else dw_advance(p, d, a.B, tiles_y, tiles_x);
    };

    auto issue = [&](const DwPos& p, int buf) {
        mbar_expect_tx(&full[buf], (uint32_t)T::BYTES);
        tma_load_4d(dsm + (size_t)buf * T::BYTES, &tmap_in, &full[buf], p.c * 64, p.x * TW * S - a.pad,
                    p.y * TH * S - a.pad, p.b);
    };

    pdl_launch_dependents();
    pdl_wait();
    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NSTAGE; s++) { mbar_init(&full[s], 1); done[s] = 0; }
        fence_barrier_init();
        tma_prefetch_desc(&tmap_in);
#pragma unroll
        for (int s = 0; s < NSTAGE; s++) {
            const int w0 = blockIdx.x + s * gridDim.x;
            if (w0 < total) issue(decompose(w0), s);
        }
    }
    __syncthreads();

    const int by = warp / (TW / BW), bx = warp % (TW / BW);     // 4 x BW output block of this warp inside the tile
    const DwPos step = decompose(gridDim.x);
    const DwPos step_ring = decompose(NSTAGE * gridDim.x);
    DwPos pos = decompose(blockIdx.x);
    const size_t out_row = (size_t)a.Wout * a.ld_out;           // elements per output image row
    int buf = 0; uint32_t phase = 0;
    int w_cblk = -1;
    float wgt[25][2];
    float bias0 = 0.f, bias1 = 0.f;
    for (int w = blockIdx.x; w < total; w += gridDim.x) {
        const int c0 = pos.c * 64 + lane * 2;
        if (pos.c != w_cblk) {                      // (re)load this lane's weights: rarely, the block index is slowest
            w_cblk = pos.c;
            const bool cok = c0 < C;
#pragma unroll
            for (int tp = 0; tp < 25; tp++) {
                const float2 wv = !cok ? make_float2(0.f, 0.f)
                                  : CBF ? *reinterpret_cast<const float2*>(s_w + (size_t)tp * C + c0)
                                        : __ldg(reinterpret_cast<const float2*>(a.weight + (size_t)tp * C + c0));
                wgt[tp][0] = wv.x; wgt[tp][1] = wv.y;
            }
            const float2 bv = !cok ? make_float2(0.f, 0.f)
                              : CBF ? *reinterpret_cast<const float2*>(s_w + 25 * (size_t)C + c0)
                                    : __ldg(reinterpret_cast<const float2*>(a.bias + c0));
            bias0 = bv.x; bias1 = bv.y;
        }
        const int oy0 = pos.y * TH + by * 4, ox0 = pos.x * TW + bx * BW;
        // every warp waits (also those whose block lies past the image edge): passing this wait proves that all
        // warps counted out of the slot's previous item, so the per-slot count never mixes two items
        mbar_wait(&full[buf], phase);
        if (oy0 < a.Hout && ox0 < a.Wout && c0 < C) {
            const unsigned char* tile = dsm + (size_t)buf * T::BYTES + lane * 4 +
                                        ((by * 4 * S) * T::IW + bx * BW * S) * 128;
            float acc[4][BW][2];
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < BW; j++) { acc[i][j][0] = bias0; acc[i][j][1] = bias1; }
#pragma unroll
            for (int ry = 0; ry < T::WIN_Y; ry++) {
                float f[T::WIN_X][2];
#pragma unroll
                for (int cx = 0; cx < T::WIN_X; cx++) {
                    const uint32_t v = *reinterpret_cast<const uint32_t*>(tile + (ry * T::IW + cx) * 128);
                    f[cx][0] = __uint_as_float(v << 16);
                    f[cx][1] = __uint_as_float(v & 0xffff0000u);
                }
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const int ky = ry - i * S;                    // compile-time after unrolling
                    if (ky < 0 || ky >= 5) continue;
#pragma unroll
                    for (int kx = 0; kx < 5; kx++) {
#pragma unroll
                        for (int j = 0; j < BW; j++) {
                            acc[i][j][0] = fmaf(f[j * S + kx][0], wgt[ky * 5 + kx][0], acc[i][j][0]);
                            acc[i][j][1] = fmaf(f[j * S + kx][1], wgt[ky * 5 + kx][1], acc[i][j][1]);
                        }
                    }
                }
            }
            if (a.relu) {
#pragma unroll
                for (int i = 0; i < 4; i++)
#pragma unroll
                    for (int j = 0; j < BW; j++) {
                        acc[i][j][0] = fmaxf(acc[i][j][0], 0.f); acc[i][j][1] = fmaxf(acc[i][j][1], 0.f);
                    }
            }
            __nv_bfloat16* orow = a.out + ((size_t)(pos.b * a.Hout + oy0) * a.Wout + ox0) * a.ld_out + a.out_col_off + c0;
            if (oy0 + 4 <= a.Hout && ox0 + BW <= a.Wout) {          // interior block: no per-pixel predicates
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    __nv_bfloat16* op = orow + i * out_row;
#pragma unroll
                    for (int j = 0; j < BW; j++)
                        *reinterpret_cast<uint32_t*>(op + (size_t)j * a.ld_out) = pack_bf16(acc[i][j][0], acc[i][j][1]);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    if (oy0 + i >= a.Hout) continue;
                    __nv_bfloat16* op = orow + i * out_row;
#pragma unroll
                    for (int j = 0; j < BW; j++) {
                        if (ox0 + j >= a.Wout) continue;
                        *reinterpret_cast<uint32_t*>(op + (size_t)j * a.ld_out) = pack_bf16(acc[i][j][0], acc[i][j][1]);
                    }
                }
            }
        }
        // count this warp out of the slot; the last one out re-arms it.  Every shared-memory read of the slot has
        // been consumed by an fma above (results are in registers), the fence orders them before the count.
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            if (atomicAdd(&done[buf], 1) == T::WARPS - 1) {
                done[buf] = 0;
                if (w + NSTAGE * (int)gridDim.x < total) {
                    DwPos pn = pos;
                    advance(pn, step_ring);
                    issue(pn, buf);
                }
            }
        }
        advance(pos, step);
        if (++buf == NSTAGE) { buf = 0; phase ^= 1; }
    }
}

// tile shapes: stride 1 -> 8x16 outputs, 4x4 blocks (8 warps, 30 KB window, 3-deep ring, 2 CTAs per SM);
//              stride 2 -> 8x16 outputs, 4x4 blocks (8 warps, 85 KB window, 2-deep ring, 1 CTA per SM): the
//              stride-2 launches are DRAM-bound on halo re-reads, the wide tile has the smaller halo (1.30x
//              against 1.41x for 8x8; measured 6.00 -> 5.88 ms over the 19 depthwise launches of a bs64 forward)
constexpr int DW1_TH = 8, DW1_TW = 16, DW2_TH = 8, DW2_TW = 16;
using DwS1 = DwTile<1, DW1_TH, DW1_TW, 4, 3>;
using DwS2 = DwTile<2, DW2_TH, DW2_TW, 4, 2>;

// ------------------------------------------------------------------ depthwise 5x5 on the tensor cores
// k_dwconv5_tma is bound by FMA issue (25 FFMA per output value, ncu: issue active 77 %), at 40 % of what HBM allows.
// The same sums as block-diagonal tcgen05 MMAs: for one tap (dy, dx) and one group of 16 channels
//     D[pixel][c] += A[pixel][c'] * B[c'][c],   A = the input window shifted by the tap, B = diag(w[tap][c])
// is ONE UMMA of M = 128 pixels, N = 16, K = 16 (8 tensor-pipe cycles at the N-proportional rate): 100 MMAs per
// 128-pixel x 64-channel item = 800 cycles, against >= 1600 cycles of FFMA for the same item.  Nothing is gathered:
// the window lies in shared memory exactly as TMA wrote it (SWIZZLE_128B, one 128-byte row per pixel = 64 channels),
// which IS the canonical K-major A layout with "row" = window pixel.  An output tile is 16 rows x 8 pixels, so the
// 8 rows of a core-matrix group are 8 horizontally consecutive window pixels and the group stride (SBO) is one
// window row; a tap only moves the descriptor start address by (dy * IW + dx) pixels = that many 128-byte rows and
// a channel group by 32 bytes inside the swizzle atom (the XOR pattern is a function of the shared-memory address).
// The depthwise weights are rounded to bf16 (as every 1x1 weight is); bias and accumulation stay f32.
// Stride 2: the window is loaded as two column-phase planes (TMA elementStrides {1,2,1,1}), so that the pixels of
// one group are again consecutive 128-byte rows; the group stride is two plane rows.
constexpr int DT_TH = 16, DT_TW = 8;
constexpr int DT_EPI_WARPS = 8;
constexpr int DT_THREADS = 64 + 32 * DT_EPI_WARPS;
constexpr int DT_B_TAP = 16 * 128;                 // one tap: 16 rows (n) x 64 k slots, diagonal of each 16x16 group
constexpr int DT_B_BYTES = 25 * DT_B_TAP;

template <int S>
struct DwTc {
    static constexpr int IH = (DT_TH - 1) * S + 5;
    static constexpr int NEED_W = (DT_TW - 1) * S + 5;                 // 12 / 19 input columns
    static constexpr int PLANES = S;
    static constexpr int PWID = S == 1 ? 12 : 10;                      // plane width in pixels
    static constexpr int PLANE_BYTES = ((IH * PWID * 128 + 1023) / 1024) * 1024;
    static constexpr int STAGE_BYTES = PLANES * PLANE_BYTES;
    static constexpr int STAGES = S == 1 ? 4 : 2;
    // stride 2 fills the 227 KB: no slack for aligning the base (the kernel traps if it is not 1024-byte aligned)
    static constexpr int SMEM = STAGES * STAGE_BYTES + DT_B_BYTES + 64 * 4 + 128 + (S == 1 ? 1024 : 0);
};

struct DwTcArgs {
    int pwid;            // plane width actually used (test switch: 12 or 16 for stride 1)
    int base_off_mode;   // test switch: 1 = put (start >> 7) & 7 into the descriptor's base-offset field
};

__device__ __forceinline__ uint64_t make_smem_desc_sbo(uint32_t smem_addr, uint32_t sbo_bytes, int base_off_mode) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3fffu);
    d |= static_cast<uint64_t>(1u) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= static_cast<uint64_t>(1u) << 46;
    if (base_off_mode) d |= static_cast<uint64_t>((smem_addr >> 7) & 7u) << 49;
    d |= static_cast<uint64_t>(2u) << 61;
    return d;
}

template <int S>
__global__ void __launch_bounds__(DT_THREADS, 1)
k_dwconv5_tc(const __grid_constant__ CUtensorMap tmap_in, DwArgs a, DwTcArgs x) {
    using T = DwTc<S>;
    extern __shared__ __align__(1024) unsigned char dt_raw[];
    unsigned char* smem = dt_raw + ((1024u - (smem_u32(dt_raw) & 1023u)) & 1023u);
    if (S == 2 && smem != dt_raw) __trap();
    const int plane_bytes = S == 1 ? ((T::IH * x.pwid * 128 + 1023) / 1024) * 1024 : T::PLANE_BYTES;
    const int stage_bytes = T::PLANES * plane_bytes;
    unsigned char* b_s = smem + (size_t)T::STAGES * stage_bytes;        // 1024-aligned: stage_bytes % 1024 == 0
    float* bias_s = reinterpret_cast<float*>(b_s + DT_B_BYTES);         // [64]
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(bias_s + 64);      // [STAGES]
    uint64_t* empty_bar = full_bar + T::STAGES;                         // [STAGES]
    uint64_t* tmem_full = empty_bar + T::STAGES;                        // [2]
    uint64_t* tmem_empty = tmem_full + 2;                               // [2]
    uint64_t* b_ready = tmem_empty + 2;                                 // [1]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_ready + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_x = (a.Wout + DT_TW - 1) / DT_TW, tiles_y = (a.Hout + DT_TH - 1) / DT_TH;
    const int cblks = (a.C8 + 7) / 8;
    const int per_c = a.B * tiles_y * tiles_x;
    const int total = per_c * cblks;
    const int C = a.C8 * 8;
    constexpr uint32_t TMEM_COLS = 128;                                 // two accumulator stages of 64 columns

    if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_in);
    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < T::STAGES; s++) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
            for (int i = 0; i < 2; i++) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], DT_EPI_WARPS); }
            mbar_init(b_ready, DT_EPI_WARPS);
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(tmem_ptr, TMEM_COLS);
    }
    // the off-diagonal zeros of B are written once; a channel-block change rewrites the diagonals only
    for (int i = tid; i < DT_B_BYTES / 16; i += DT_THREADS) reinterpret_cast<uint4*>(b_s)[i] = make_uint4(0, 0, 0, 0);
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    pdl_launch_dependents();
    pdl_wait();

    const DwPos step = dw_decompose(gridDim.x, per_c, tiles_y, tiles_x);
    DwPos pos = dw_decompose(blockIdx.x, per_c, tiles_y, tiles_x);

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int w = blockIdx.x; w < total; w += gridDim.x) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                unsigned char* dst = smem + (size_t)stage * stage_bytes;
                const int x0 = pos.x * DT_TW * S - a.pad, y0 = pos.y * DT_TH * S - a.pad;
                mbar_expect_tx(&full_bar[stage], (uint32_t)(T::PLANES * T::IH * x.pwid * 128));
#pragma unroll
                for (int p = 0; p < T::PLANES; p++)
                    tma_load_4d(dst + (size_t)p * plane_bytes, &tmap_in, &full_bar[stage], pos.c * 64, x0 + p, y0, pos.b);
                dw_advance(pos, step, a.B, tiles_y, tiles_x);
                if (++stage == T::STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp runs the loop converged (descriptor arithmetic on the uniform datapath),
        // one elected lane issues =====
        {
            const uint32_t idesc = make_instr_desc(BM, 16);
            const uint32_t sbo = (uint32_t)(S * x.pwid * 128);              // one output row down = S plane rows
            const uint32_t a_hi = (uint32_t)(make_smem_desc_sbo(0, sbo, 0) >> 32);
            const uint32_t b_hi = (uint32_t)(make_smem_desc(0) >> 32);
            const uint32_t b_lo0 = (smem_u32(b_s) >> 4) | (1u << 16);
            const uint32_t tmem_b = __shfl_sync(0xffffffffu, tmem_base, 0);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            int cur_c = -1; uint32_t b_phase = 0;
            for (int w = blockIdx.x; w < total; w += gridDim.x) {
                if (pos.c != cur_c) {                                        // weights of a new channel block
                    cur_c = pos.c;
                    mbar_wait(b_ready, b_phase); b_phase ^= 1;
                }
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                mbar_wait(&full_bar[stage], phase);
                __syncwarp();
                tcgen05_fence_after();
                const uint32_t sa = smem_u32(smem) + (uint32_t)(stage * stage_bytes);
                const uint32_t a_lo0 = (sa >> 4) | (1u << 16);
                const uint32_t d_tmem = tmem_b + (uint32_t)(acc * 64);
#pragma unroll 1
                for (int dy = 0; dy < 5; dy++) {
                    const uint32_t a_row = a_lo0 + (uint32_t)(dy * x.pwid * 8);
                    const uint32_t b_row = b_lo0 + (uint32_t)(dy * 5 * (DT_B_TAP >> 4));
#pragma unroll
                    for (int dx = 0; dx < 5; dx++) {
                        const uint32_t a_tap = a_row + (uint32_t)((dx % S) * (plane_bytes >> 4)) + (uint32_t)((dx / S) * 8);
                        const uint32_t b_tap = b_row + (uint32_t)(dx * (DT_B_TAP >> 4));
#pragma unroll
                        for (int gq = 0; gq < 4; gq++) {
                            uint32_t ahi = a_hi;
                            if (x.base_off_mode) ahi |= (((a_tap + gq * 2) >> 3) & 7u) << 17;
                            umma_bf16_elect(d_tmem + (uint32_t)(gq * 16), a_tap + gq * 2, ahi, b_tap + gq * 2, b_hi, idesc,
                                            (dy | dx) != 0 ? 1u : 0u);
                        }
                    }
                }
                umma_commit_elect(&empty_bar[stage]);
                umma_commit_elect(&tmem_full[acc]);
                dw_advance(pos, step, a.B, tiles_y, tiles_x);
                if (++stage == T::STAGES) { stage = 0; phase ^= 1; }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue warps: TMEM lane quadrant = warp % 4, column half = (warp - 2) / 4 =====
        const int q = warp & 3, half = (warp - 2) >> 2;
        const int etid = tid - 64;
        const int row = q * 32 + lane;                      // tile row == TMEM lane: output pixel (row / 8, row % 8)
        const int ry = row / DT_TW, rx = row % DT_TW;
        int acc = 0; uint32_t acc_phase = 0;
        int cur_c = -1;
        for (int w = blockIdx.x; w < total; w += gridDim.x) {
            if (pos.c != cur_c) {
                // every MMA that read the old diagonals has retired: this warp has passed tmem_full of all earlier
                // items, and the issuer does not start this item before b_ready
                cur_c = pos.c;
                for (int i = etid; i < 25 * 64; i += 32 * DT_EPI_WARPS) {
                    const int tap = i >> 6, c = i & 63, gq = c >> 4, n = c & 15;
                    const int cg = pos.c * 64 + c;
                    const float wv = cg < C ? a.weight[(size_t)tap * C + cg] : 0.f;
                    const int chunk = 2 * gq + (n >> 3);
                    *reinterpret_cast<__nv_bfloat16*>(b_s + tap * DT_B_TAP + n * 128 + ((chunk ^ (n & 7)) << 4) + (n & 7) * 2) =
                        __float2bfloat16_rn(wv);
                }
                // bias_s is read by the epilogue warps only: order the rewrite behind their reads of the old values
                asm volatile("bar.sync 1, %0;" ::"n"(32 * DT_EPI_WARPS) : "memory");
                if (etid < 64) bias_s[etid] = pos.c * 64 + etid < C ? a.bias[pos.c * 64 + etid] : 0.f;
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                asm volatile("bar.sync 1, %0;" ::"n"(32 * DT_EPI_WARPS) : "memory");
                if (lane == 0) mbar_arrive(b_ready);
            }
            mbar_wait(&tmem_full[acc], acc_phase);
            tcgen05_fence_after();
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (uint32_t)(acc * 64 + half * 32);
            uint32_t va[CHUNK], vb[CHUNK];
            tmem_ld16_async(t_row, va);
            tmem_ld16_async(t_row + 16, vb);
            tmem_ld_wait(va);
            tmem_ld_wait(vb);
            // the accumulator stage is free as soon as its values are in registers
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            const int oy = pos.y * DT_TH + ry, ox = pos.x * DT_TW + rx;
            const int c0 = pos.c * 64 + half * 32;
            if (oy < a.Hout && ox < a.Wout) {
                __nv_bfloat16* op = a.out + ((size_t)(pos.b * a.Hout + oy) * a.Wout + ox) * a.ld_out + a.out_col_off + c0;
                const float* bs = bias_s + half * 32;
#pragma unroll
                for (int h8 = 0; h8 < 4; h8++) {
                    if (c0 + h8 * 8 >= C) break;
                    const uint32_t* v = h8 < 2 ? va + h8 * 8 : vb + (h8 - 2) * 8;
                    float f[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        f[j] = __uint_as_float(v[j]) + bs[h8 * 8 + j];
                        if (a.relu) f[j] = fmaxf(f[j], 0.f);
                    }
                    uint4 ov;
                    ov.x = pack_bf16(f[0], f[1]); ov.y = pack_bf16(f[2], f[3]);
                    ov.z = pack_bf16(f[4], f[5]); ov.w = pack_bf16(f[6], f[7]);
                    *reinterpret_cast<uint4*>(op + h8 * 8) = ov;
                }
            }
            dw_advance(pos, step, a.B, tiles_y, tiles_x);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// generic depthwise kxk (any kernel/stride): one output pixel x 8 channels per thread
__global__ void __launch_bounds__(256) k_dwconv(DwArgs a) {
    const long long total = (long long)a.B * a.Hout * a.Wout * a.C8;
    const int C = a.C8 * 8;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        const int c8 = (int)(t % a.C8);
        long long p = t / a.C8;
        const int ox = (int)(p % a.Wout); p /= a.Wout;
        const int oy = (int)(p % a.Hout);
        const int b = (int)(p / a.Hout);
        float acc[8];
        const float4 b0 = *reinterpret_cast<const float4*>(a.bias + c8 * 8);
        const float4 b1 = *reinterpret_cast<const float4*>(a.bias + c8 * 8 + 4);
        acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w;
        acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
        for (int ky = 0; ky < a.kernel; ky++) {
            const int iy = oy * a.stride - a.pad + ky;
            if (iy < 0 || iy >= a.Hin) continue;
            for (int kx = 0; kx < a.kernel; kx++) {
                const int ix = ox * a.stride - a.pad + kx;
                if (ix < 0 || ix >= a.Win) continue;
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(
                    a.in + ((size_t)(b * a.Hin + iy) * a.Win + ix) * a.ld_in + a.in_col_off + c8 * 8));
                const float* wp = a.weight + (size_t)(ky * a.kernel + kx) * C + c8 * 8;
                const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
                const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
                const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
                const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]);
                const float2 f2 = __bfloat1622float2(h[2]), f3 = __bfloat1622float2(h[3]);
                acc[0] = fmaf(f0.x, w0.x, acc[0]); acc[1] = fmaf(f0.y, w0.y, acc[1]);
                acc[2] = fmaf(f1.x, w0.z, acc[2]); acc[3] = fmaf(f1.y, w0.w, acc[3]);
                acc[4] = fmaf(f2.x, w1.x, acc[4]); acc[5] = fmaf(f2.y, w1.y, acc[5]);
                acc[6] = fmaf(f3.x, w1.z, acc[6]); acc[7] = fmaf(f3.y, w1.w, acc[7]);
            }
        }
        if (a.relu) {
#pragma unroll
            for (int j = 0; j < 8; j++) acc[j] = fmaxf(acc[j], 0.f);
        }
        uint4 o;
        o.x = pack_bf16(acc[0], acc[1]); o.y = pack_bf16(acc[2], acc[3]);
        o.z = pack_bf16(acc[4], acc[5]); o.w = pack_bf16(acc[6], acc[7]);
        *reinterpret_cast<uint4*>(a.out + ((size_t)(b * a.Hout + oy) * a.Wout + ox) * a.ld_out + a.out_col_off + c8 * 8) = o;
    }
}


// Depthwise kxk (k = 3 or 5, stride 1 or 2) of the MobileNet blocks (torchvision InvertedResidual behind
// basenetworks.py:407-458) with any fused activation code, on any channel count in 8-channel groups: the TMA kernels
// above work on 64-channel items, which on the 16..72-channel tensors at 641^2 and 321^2 would spend most of their
// shared memory and FMAs on fill.  One thread = 8 channels x DW_OX consecutive output pixels of one row, register
// blocked like k_dwconv5.  Per image the items run channel group fastest, then the strip, then the row, so a warp
// reads whole input rows.  CTA = (chunk of NIT * blockDim items, image); blockDim is a multiple of C8, so a thread
// keeps its channel group over all its items.
// Squeeze-excitation blocks (se_part != nullptr): the CTA also writes the sums of its f32 post-activation outputs per
// channel to slot [image][chunk][channel], reduced in a fixed order without atomics -- deterministic, and independent
// of the batch (the chunking depends on the image size only).  k_se reduces the slots.
struct DwNcArgs { float* se_part; int nit, nslots; };

template <int K, int S>
__global__ void __launch_bounds__(256) k_dwconv_nc(DwArgs a, DwNcArgs x) {
    constexpr int NCOL = (DW_OX - 1) * S + K;
    const int b = blockIdx.y;
    const int strips = (a.Wout + DW_OX - 1) / DW_OX;
    const int per_img = a.Hout * strips * a.C8;
    const int C = a.C8 * 8;
    const int c8 = threadIdx.x % a.C8;
    float sum[8];
#pragma unroll
    for (int j = 0; j < 8; j++) sum[j] = 0.f;
    float bias[8];
    {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(a.bias + c8 * 8));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(a.bias + c8 * 8 + 4));
        bias[0] = b0.x; bias[1] = b0.y; bias[2] = b0.z; bias[3] = b0.w;
        bias[4] = b1.x; bias[5] = b1.y; bias[6] = b1.z; bias[7] = b1.w;
    }
    const int t0 = blockIdx.x * blockDim.x * x.nit + threadIdx.x;
    for (int it = 0; it < x.nit; it++) {
        const int t = t0 + it * blockDim.x;
        if (t >= per_img) break;
        const int p = t / a.C8;
        const int sx = p % strips, oy = p / strips;
        const int ox0 = sx * DW_OX;
        const int ix0 = ox0 * S - a.pad;
        float acc[DW_OX][8];
#pragma unroll
        for (int o = 0; o < DW_OX; o++)
#pragma unroll
            for (int j = 0; j < 8; j++) acc[o][j] = bias[j];
#pragma unroll
        for (int ky = 0; ky < K; ky++) {
            const int iy = oy * S - a.pad + ky;
            if (iy < 0 || iy >= a.Hin) continue;
            float w[K][8];
#pragma unroll
            for (int kx = 0; kx < K; kx++) {
                const float* wp = a.weight + (size_t)(ky * K + kx) * C + c8 * 8;
                const float4 w0 = __ldg(reinterpret_cast<const float4*>(wp));
                const float4 w1 = __ldg(reinterpret_cast<const float4*>(wp + 4));
                w[kx][0] = w0.x; w[kx][1] = w0.y; w[kx][2] = w0.z; w[kx][3] = w0.w;
                w[kx][4] = w1.x; w[kx][5] = w1.y; w[kx][6] = w1.z; w[kx][7] = w1.w;
            }
            const __nv_bfloat16* rowp = a.in + ((size_t)(b * a.Hin + iy) * a.Win) * a.ld_in + a.in_col_off + c8 * 8;
#pragma unroll
            for (int col = 0; col < NCOL; col++) {
                const int ix = ix0 + col;
                if (ix < 0 || ix >= a.Win) continue;
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(rowp + (size_t)ix * a.ld_in));
                float f[8];
                unpack8(v, f);
#pragma unroll
                for (int o = 0; o < DW_OX; o++) {
                    const int kx = col - o * S;       // compile-time after unrolling
                    if (kx < 0 || kx >= K) continue;
#pragma unroll
                    for (int j = 0; j < 8; j++) acc[o][j] = fmaf(f[j], w[kx][j], acc[o][j]);
                }
            }
        }
#pragma unroll
        for (int o = 0; o < DW_OX; o++) {
            const int ox = ox0 + o;
            if (ox >= a.Wout) continue;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                acc[o][j] = act_f(acc[o][j], a.relu);
                sum[j] += acc[o][j];
            }
            uint4 ov;
            ov.x = pack_bf16(acc[o][0], acc[o][1]); ov.y = pack_bf16(acc[o][2], acc[o][3]);
            ov.z = pack_bf16(acc[o][4], acc[o][5]); ov.w = pack_bf16(acc[o][6], acc[o][7]);
            *reinterpret_cast<uint4*>(a.out + ((size_t)(b * a.Hout + oy) * a.Wout + ox) * a.ld_out + a.out_col_off + c8 * 8) = ov;
        }
    }
    if (x.se_part == nullptr) return;
    __shared__ float s_sum[256][9];
#pragma unroll
    for (int j = 0; j < 8; j++) s_sum[threadIdx.x][j] = sum[j];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const int g = c >> 3, j = c & 7;
        float v = 0.f;
        for (int t = g; t < (int)blockDim.x; t += a.C8) v += s_sum[t][j];
        x.se_part[((size_t)b * x.nslots + blockIdx.x) * C + c] = v;
    }
}

// torchvision SqueezeExcitation (avg-pool -> fc1 -> ReLU -> fc2 -> Hardsigmoid -> x * s) folded into the weights of
// the projection 1x1 that follows it: one CTA per image reduces the depthwise kernel's channel-sum slots in a fixed
// order, runs the two small FCs and writes that image's projection weights bf16(W[n][k] * s[k]) in the B layout of
// the implicit-GEMM conv (kernel 1), which then reads the rows of its image (GemmArgs::w_img_rows).
struct SeArgs {
    const float* part; int nslots, C8;      // [B][nslots][C8 * 8] channel sums (k_dwconv_nc)
    float inv_hw;                           // 1 / (pixels of the depthwise output)
    int channels, squeeze;
    const float *w1, *b1, *w2, *b2;         // fc1 [squeeze][channels] + [squeeze], fc2 [channels][squeeze] + [channels]
    const float* wproj;                     // f32 [n_pad][k_total] projection weights (folded BN), zero padded
    int n_pad, k_total;
    __nv_bfloat16* wimg;                    // [max_batch][n_pad][k_total]
};

constexpr int SE_THREADS = 512;

__global__ void __launch_bounds__(SE_THREADS) k_se(SeArgs a) {
    extern __shared__ float se_s[];         // pooled [C], hidden [squeeze], scale [C]
    const int b = blockIdx.x, C = a.C8 * 8;
    float* pooled = se_s;
    float* hid = se_s + C;
    float* sc = hid + a.squeeze;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float* p = a.part + (size_t)b * a.nslots * C + c;
        float v = 0.f;
        for (int i = 0; i < a.nslots; i++) v += p[(size_t)i * C];
        pooled[c] = v * a.inv_hw;
    }
    __syncthreads();
    for (int j = threadIdx.x; j < a.squeeze; j += blockDim.x) {
        float h = a.b1[j];
        const float* w = a.w1 + (size_t)j * a.channels;
        for (int c = 0; c < a.channels; c++) h = fmaf(w[c], pooled[c], h);
        hid[j] = fmaxf(h, 0.f);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float s = 0.f;
        if (c < a.channels) {
            float v = a.b2[c];
            const float* w = a.w2 + (size_t)c * a.squeeze;
            for (int j = 0; j < a.squeeze; j++) v = fmaf(w[j], hid[j], v);
            s = fminf(fmaxf(v + 3.f, 0.f), 6.f) / 6.f;      // torch.nn.Hardsigmoid
        }
        sc[c] = s;
    }
    __syncthreads();
    const int n_w = a.n_pad * a.k_total;
    __nv_bfloat16* out = a.wimg + (size_t)b * n_w;
    for (int i = threadIdx.x; i < n_w; i += blockDim.x) {
        const int k = i % a.k_total;
        out[i] = __float2bfloat16_rn(a.wproj[i] * (k < C ? sc[k] : 0.f));
    }
}

// ------------------------------------------------------------------ fused depthwise 5x5 -> 1x1 GEMM
// InvertedResidualK branch2 tail (basenetworks.py:219-226: dw5x5, BN, 1x1, BN, ReLU) as ONE kernel: the depthwise
// output never visits HBM.  Per CTA (persistent over 8 x 16 output-pixel patches == 128-row M tiles), per 64-channel
// K block:
//   warp 0     TMA producer: the patch's input window (12 x 20 pixels x 64 channels, zero fill == conv padding) into
//              a window ring, and the K block of the 1x1 weights [n_pad x 64] into a B ring
//   warps 2-9  depthwise: one warp = a 4 x 4 block of output pixels, one lane = a channel pair (the register-blocked
//              FMA loop of k_dwconv5_tma); results go as bf16 straight into a 128B-swizzled K-major A stage
//              (row = pixel of the patch, the layout TMA would have produced), fence.proxy.async + mbarrier arrive
//   warp 1     tcgen05.mma issuer: D[128 x n_pad] += A-stage x B-stage^T in TMEM; tcgen05.commit frees the stages
//   warps 10-13 epilogue: TMEM -> registers -> bias + ReLU -> bf16 -> scatter / plain stores (epilogue_chunk)
// n_pad <= 512 TMEM columns; n_pad > 256 runs as two UMMA halves; two accumulator stages when 2 * n_pad <= 512.
constexpr int FD_DW_WARPS = 8, FD_EPI_WARPS = 4;
constexpr int FD_THREADS = 32 * (2 + FD_DW_WARPS + FD_EPI_WARPS);     // 448

struct FusedArgs {
    const float* dw_weight;      // [25][C] f32, tap-major
    const float* dw_bias;        // [C]
    int C;                       // physical channels of the depthwise input (multiple of 8)
    int dw_relu, pad;
    int ws, as, bs;              // ring depths: windows, A stages, B stages
    int n_pad, n_halves, half_n; // n_pad = n_halves * half_n, half_n <= 256, multiple of 16
    int acc_stages;
};

__device__ __forceinline__ void fence_proxy_async_shared() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <int S>
__global__ void __launch_bounds__(FD_THREADS, 1)
k_dw_gemm(const __grid_constant__ CUtensorMap tmap_win, const __grid_constant__ CUtensorMap tmap_b, GemmArgs g, FusedArgs f) {
    using T = DwTile<S, PH, PW, 4, 1>;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int a_bytes = BM * BK * 2;                     // 16 KB
    const int b_bytes = f.n_pad * BK * 2;                // multiple of 1024 (n_pad % 16 == 0)
    unsigned char* a_st = smem;
    unsigned char* b_st = a_st + (size_t)f.as * a_bytes;
    unsigned char* win = b_st + (size_t)f.bs * b_bytes;
    float* bias_s = reinterpret_cast<float*>(win + (size_t)f.ws * T::BYTES);
    DestGroup* dest_s = reinterpret_cast<DestGroup*>(bias_s + f.n_pad);
    // depthwise weights [25][C] + bias [C], staged once per CTA: a per-K-block reload from global memory put the
    // depthwise warps on the long scoreboard (ncu round 2: 1.4 - 2.8 warps per issue, the L1 is carved down to a few KB)
    float* dww_s = reinterpret_cast<float*>(dest_s + f.n_pad / CHUNK);
    uint64_t* bars = reinterpret_cast<uint64_t*>(dww_s + 26 * (size_t)f.C);
    uint64_t* win_full = bars;                 uint64_t* win_empty = win_full + f.ws;
    uint64_t* a_full = win_empty + f.ws;       uint64_t* a_empty = a_full + f.as;
    uint64_t* b_full = a_empty + f.as;         uint64_t* b_empty = b_full + f.bs;
    uint64_t* tmem_full = b_empty + f.bs;      uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t need_cols = (uint32_t)(f.acc_stages * f.n_pad);
    const uint32_t tmem_cols = need_cols <= 32 ? 32 : need_cols <= 64 ? 64 : need_cols <= 128 ? 128 : need_cols <= 256 ? 256 : 512;

    if (warp == 0 && lane == 0) { tma_prefetch_desc(&tmap_win); tma_prefetch_desc(&tmap_b); }
    for (int i = threadIdx.x; i < f.n_pad; i += FD_THREADS) bias_s[i] = g.bias[i];
    if (g.mode == MODE_SCATTER)
        for (int i = threadIdx.x; i < f.n_pad / CHUNK; i += FD_THREADS) dest_s[i] = g.dest[i];
    for (int i = threadIdx.x; i < 25 * f.C; i += FD_THREADS) dww_s[i] = f.dw_weight[i];
    for (int i = threadIdx.x; i < f.C; i += FD_THREADS) dww_s[25 * f.C + i] = f.dw_bias[i];
    if (warp == 1) {
        if (lane == 0) {
            for (int i = 0; i < f.ws; i++) { mbar_init(&win_full[i], 1); mbar_init(&win_empty[i], FD_DW_WARPS); }
            for (int i = 0; i < f.as; i++) { mbar_init(&a_full[i], FD_DW_WARPS); mbar_init(&a_empty[i], 1); }
            for (int i = 0; i < f.bs; i++) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
            for (int i = 0; i < 2; i++) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], FD_EPI_WARPS); }
            fence_barrier_init();
        }
        __syncwarp();
        tmem_alloc(tmem_ptr, tmem_cols);
    }
    tcgen05_fence_before();
    __syncthreads();
    tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    // (after the TMEM allocation: a dependent CTA that becomes co-resident must not take the columns first)
    pdl_launch_dependents();
    pdl_wait();
    const int per_img = g.tiles_x * g.tiles_y;
    const int nkb = g.num_k_blocks;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int wi = 0; uint32_t wph = 0; int bi = 0; uint32_t bph = 0;
            for (int tile = blockIdx.x; tile < g.m_blocks; tile += gridDim.x) {
                const int img = tile / per_img, t = tile - img * per_img;
                const int cy = (t / g.tiles_x) * PH * S - f.pad, cx = (t % g.tiles_x) * PW * S - f.pad;
                for (int kb = 0; kb < nkb; kb++) {
                    mbar_wait(&win_empty[wi], wph ^ 1);
                    mbar_expect_tx(&win_full[wi], (uint32_t)T::BYTES);
                    tma_load_4d(win + (size_t)wi * T::BYTES, &tmap_win, &win_full[wi], kb * 64, cx, cy, img);
                    if (++wi == f.ws) { wi = 0; wph ^= 1; }
                    mbar_wait(&b_empty[bi], bph ^ 1);
                    mbar_expect_tx(&b_full[bi], (uint32_t)b_bytes);
                    for (int h = 0; h < f.n_halves; h++)
                        tma_load_2d(b_st + (size_t)bi * b_bytes + (size_t)h * f.half_n * BK * 2, &tmap_b, &b_full[bi],
                                    kb * BK, h * f.half_n);
                    if (++bi == f.bs) { bi = 0; bph ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            const uint32_t idesc = make_instr_desc(BM, f.half_n);
            int ai = 0; uint32_t aph = 0; int bi = 0; uint32_t bph = 0; int acc = 0; uint32_t acc_ph = 0;
            for (int tile = blockIdx.x; tile < g.m_blocks; tile += gridDim.x) {
                mbar_wait(&tmem_empty[acc], acc_ph ^ 1);
                tcgen05_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * f.n_pad);
                for (int kb = 0; kb < nkb; kb++) {
                    mbar_wait(&a_full[ai], aph);
                    mbar_wait(&b_full[bi], bph);
                    tcgen05_fence_after();
                    const uint32_t sa = smem_u32(a_st + (size_t)ai * a_bytes);
                    const uint32_t sb = smem_u32(b_st + (size_t)bi * b_bytes);
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; k++) {
                        const uint64_t adesc = make_smem_desc(sa + k * UMMA_K * 2);
                        for (int h = 0; h < f.n_halves; h++) {
                            const uint64_t bdesc = make_smem_desc(sb + (uint32_t)(h * f.half_n * BK * 2) + k * UMMA_K * 2);
                            umma_bf16(d_tmem + (uint32_t)(h * f.half_n), adesc, bdesc, idesc, (kb | k) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(&a_empty[ai]);
                    umma_commit(&b_empty[bi]);
                    if (++ai == f.as) { ai = 0; aph ^= 1; }
                    if (++bi == f.bs) { bi = 0; bph ^= 1; }
                }
                umma_commit(&tmem_full[acc]);
                if (++acc == f.acc_stages) { acc = 0; acc_ph ^= 1; }
            }
        }
    } else if (warp < 2 + FD_DW_WARPS) {
        // ===== depthwise warps =====
        const int dwi = warp - 2;
        const int by = dwi / (PW / 4), bx = dwi % (PW / 4);        // 4 x 4 output block of this warp inside the patch
        int wi = 0; uint32_t wph = 0; int ai = 0; uint32_t aph = 0;
        for (int tile = blockIdx.x; tile < g.m_blocks; tile += gridDim.x) {
            const int img = tile / per_img, t = tile - img * per_img;
            const int oy0 = (t / g.tiles_x) * PH + by * 4, ox0 = (t % g.tiles_x) * PW + bx * 4;
            const bool inside = oy0 < g.Ho && ox0 < g.Wo;            // blocks past the image edge: rows nobody stores
            (void)img;
            for (int kb = 0; kb < nkb; kb++) {
                const int c0 = kb * 64 + lane * 2;
                const bool cok = c0 < f.C;
                float wgt[25][2];
                float bias0 = 0.f, bias1 = 0.f;
                if (inside) {
#pragma unroll
                    for (int tp = 0; tp < 25; tp++) {
                        const float2 wv = cok ? *reinterpret_cast<const float2*>(dww_s + (size_t)tp * f.C + c0)
                                              : make_float2(0.f, 0.f);
                        wgt[tp][0] = wv.x; wgt[tp][1] = wv.y;
                    }
                    if (cok) { const float2 bv = *reinterpret_cast<const float2*>(dww_s + 25 * (size_t)f.C + c0); bias0 = bv.x; bias1 = bv.y; }
                }
                float acc[4][4][2];
                mbar_wait(&win_full[wi], wph);
                if (inside) {
                    const unsigned char* tile_p = win + (size_t)wi * T::BYTES + lane * 4 +
                                                  ((by * 4 * S) * T::IW + bx * 4 * S) * 128;
#pragma unroll
                    for (int i = 0; i < 4; i++)
#pragma unroll
                        for (int j = 0; j < 4; j++) { acc[i][j][0] = bias0; acc[i][j][1] = bias1; }
#pragma unroll
                    for (int ry = 0; ry < T::WIN_Y; ry++) {
                        float v2[T::WIN_X][2];
#pragma unroll
                        for (int cx = 0; cx < T::WIN_X; cx++) {
                            const uint32_t v = *reinterpret_cast<const uint32_t*>(tile_p + (ry * T::IW + cx) * 128);
                            v2[cx][0] = __uint_as_float(v << 16);
                            v2[cx][1] = __uint_as_float(v & 0xffff0000u);
                        }
#pragma unroll
                        for (int i = 0; i < 4; i++) {
                            const int ky = ry - i * S;                    // compile-time after unrolling
                            if (ky < 0 || ky >= 5) continue;
#pragma unroll
                            for (int kx = 0; kx < 5; kx++) {
#pragma unroll
                                for (int j = 0; j < 4; j++) {
                                    acc[i][j][0] = fmaf(v2[j * S + kx][0], wgt[ky * 5 + kx][0], acc[i][j][0]);
                                    acc[i][j][1] = fmaf(v2[j * S + kx][1], wgt[ky * 5 + kx][1], acc[i][j][1]);
                                }
                            }
                        }
                    }
                    if (f.dw_relu) {
#pragma unroll
                        for (int i = 0; i < 4; i++)
#pragma unroll
                            for (int j = 0; j < 4; j++) {
                                acc[i][j][0] = fmaxf(acc[i][j][0], 0.f); acc[i][j][1] = fmaxf(acc[i][j][1], 0.f);
                            }
                    }
                }
                // the window slot is free as soon as its values sit in registers
                __syncwarp();
                if (lane == 0) mbar_arrive(&win_empty[wi]);
                if (++wi == f.ws) { wi = 0; wph ^= 1; }
                // A stage: row = pixel of the patch, 16-byte chunk index XOR (row & 7) (SWIZZLE_128B, K-major)
                mbar_wait(&a_empty[ai], aph ^ 1);
                if (inside) {
                    unsigned char* a_base = a_st + (size_t)ai * a_bytes + (lane & 3) * 4;
#pragma unroll
                    for (int i = 0; i < 4; i++)
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const int row = (by * 4 + i) * PW + bx * 4 + j;
                            *reinterpret_cast<uint32_t*>(a_base + row * 128 + ((((lane >> 2) ^ (row & 7))) << 4)) =
                                pack_bf16(acc[i][j][0], acc[i][j][1]);
                        }
                }
                fence_proxy_async_shared();
                __syncwarp();
                if (lane == 0) mbar_arrive(&a_full[ai]);
                if (++ai == f.as) { ai = 0; aph ^= 1; }
            }
        }
    } else {
        // ===== epilogue warps: TMEM lane quadrant = warp % 4 =====
        const int q = warp & 3;
        const int n_chunks = f.n_pad / CHUNK;
        int acc = 0; uint32_t acc_ph = 0;
        for (int tile = blockIdx.x; tile < g.m_blocks; tile += gridDim.x) {
            mbar_wait(&tmem_full[acc], acc_ph);
            tcgen05_fence_after();
            const int m = tile_row_to_m(g, tile, q * 32 + lane);
            const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (uint32_t)(acc * f.n_pad);
            uint32_t va[CHUNK], vb[CHUNK];
            auto process = [&](int ci, const uint32_t* v) {
                float accf[CHUNK];
#pragma unroll
                for (int j = 0; j < CHUNK; j++) accf[j] = __uint_as_float(v[j]);
                const int n0 = ci * CHUNK;
                if (n0 < ((g.N + 7) & ~7)) epilogue_chunk<false>(g, m, n0, accf, bias_s + n0, nullptr, dest_s);
            };
            tmem_ld16_async(t_row, va);
            for (int ci = 0; ci < n_chunks; ci += 2) {
                tmem_ld_wait(va);
                if (ci + 1 < n_chunks) tmem_ld16_async(t_row + (uint32_t)((ci + 1) * CHUNK), vb);
                process(ci, va);
                if (ci + 1 < n_chunks) {
                    tmem_ld_wait(vb);
                    if (ci + 2 < n_chunks) tmem_ld16_async(t_row + (uint32_t)((ci + 2) * CHUNK), va);
                    process(ci + 1, vb);
                }
            }
            tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == f.acc_stages) { acc = 0; acc_ph ^= 1; }
        }
    }
    tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        tcgen05_fence_after();
        tmem_dealloc(tmem_base, tmem_cols);
    }
}

size_t fused_smem_bytes(int ws, int as, int bs, int n_pad, int c_dw) {
    return 1024 + (size_t)as * BM * BK * 2 + (size_t)bs * n_pad * BK * 2 + (size_t)ws * DwTile<1, PH, PW, 4, 1>::BYTES +
           (size_t)n_pad * 5 + (size_t)c_dw * 26 * 4 + (size_t)(2 * (ws + as + bs) + 4) * 8 + 64;
}

// ------------------------------------------------------------------ input conv: f32 NCHW [B,3,H,W] -> bf16 NHWC
struct InConvArgs {
    const float* in; __nv_bfloat16* out; int ld_out;
    // raw-image variant: uint8 [B][H][W][3] (what PIL / the decoder of a video stream delivers); the kernel applies
    // torchvision's ToTensor + Normalize (transforms/__init__.py:26-33) on load: ((u / 255) - mean[c]) / std[c]
    const uint8_t* in_u8; float mean[3], stdev[3];
    const float* weight;   // [3*k*k][C8*8] (tap-major)
    const float* bias;     // [C8*8]
    int B, Hin, Win, Hout, Wout, C8, kernel, stride, pad, relu;
};

// EXT: activation codes 2 / 3 (the MobileNet stems); EXT = false is the ReLU-only kernel of the other backbones
template <int KS, bool U8, bool EXT = false>
__global__ void __launch_bounds__(256) k_input_conv(InConvArgs a) {
    // one thread = one output pixel, all output channels: the 3*k*k input samples are loaded once (registers for
    // k = 3, thread-local memory for k = 7) and reused for every 8-channel group; weights are broadcast reads
    // from shared memory
    extern __shared__ __align__(16) float s_w[];      // [3*k*k][C] weights + [C] bias
    constexpr int TAPS = 3 * KS * KS;
    const int C = a.C8 * 8;
    const int n_w = TAPS * C;
    for (int i = threadIdx.x; i < n_w; i += blockDim.x) s_w[i] = a.weight[i];
    for (int i = threadIdx.x; i < C; i += blockDim.x) s_w[n_w + i] = a.bias[i];
    // raw images: the 256 possible values of a channel, normalised once per CTA with IEEE division / subtraction
    // (bit-identical to torchvision's ToTensor + Normalize on the host) -> one byte load + one table read per sample
    float* s_lut = s_w + n_w + C;                     // [3][256]
    if (U8)
        for (int i = threadIdx.x; i < 256; i += blockDim.x) {
            const float x = __fdiv_rn((float)i, 255.f);
#pragma unroll
            for (int c = 0; c < 3; c++) s_lut[c * 256 + i] = __fdiv_rn(__fsub_rn(x, a.mean[c]), a.stdev[c]);
        }
    pdl_launch_dependents();
    pdl_wait();
    __syncthreads();
    const long long total = (long long)a.B * a.Hout * a.Wout;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;
         t += (long long)gridDim.x * blockDim.x) {
        long long p = t;
        const int ox = (int)(p % a.Wout); p /= a.Wout;
        const int oy = (int)(p % a.Hout);
        const int b = (int)(p / a.Hout);
        float in[TAPS];
        if (U8) {
            // HWC bytes: the three channels of a pixel are adjacent; one row pointer per ky, one pixel pointer per kx
#pragma unroll
            for (int ky = 0; ky < KS; ky++) {
                const int iy = oy * a.stride - a.pad + ky;
                const bool oky = iy >= 0 && iy < a.Hin;
                const uint8_t* rowp = a.in_u8 + ((size_t)b * a.Hin + (oky ? iy : 0)) * a.Win * 3;
#pragma unroll
                for (int kx = 0; kx < KS; kx++) {
                    const int ix = ox * a.stride - a.pad + kx;
                    const bool ok = oky && ix >= 0 && ix < a.Win;
                    const uint8_t* px = rowp + (ok ? ix : 0) * 3;
#pragma unroll
                    for (int ci = 0; ci < 3; ci++)
                        in[(ci * KS + ky) * KS + kx] = ok ? s_lut[ci * 256 + __ldg(px + ci)] : 0.f;
                }
            }
        } else {
#pragma unroll
            for (int ci = 0; ci < 3; ci++) {
                const float* plane = a.in + ((size_t)b * 3 + ci) * a.Hin * a.Win;
#pragma unroll
                for (int ky = 0; ky < KS; ky++) {
                    const int iy = oy * a.stride - a.pad + ky;
#pragma unroll
                    for (int kx = 0; kx < KS; kx++) {
                        const int ix = ox * a.stride - a.pad + kx;
                        const bool ok = iy >= 0 && iy < a.Hin && ix >= 0 && ix < a.Win;
                        in[(ci * KS + ky) * KS + kx] = ok ? __ldg(plane + (size_t)iy * a.Win + ix) : 0.f;
                    }
                }
            }
        }
        __nv_bfloat16* orow = a.out + ((size_t)(b * a.Hout + oy) * a.Wout + ox) * a.ld_out;
        for (int c8 = 0; c8 < a.C8; c8++) {
            float acc[8];
            const float4 b0 = *reinterpret_cast<const float4*>(s_w + n_w + c8 * 8);
            const float4 b1 = *reinterpret_cast<const float4*>(s_w + n_w + c8 * 8 + 4);
            acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w;
            acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
#pragma unroll
            for (int tp = 0; tp < TAPS; tp++) {
                const float4 w0 = *reinterpret_cast<const float4*>(s_w + (size_t)tp * C + c8 * 8);
                const float4 w1 = *reinterpret_cast<const float4*>(s_w + (size_t)tp * C + c8 * 8 + 4);
                const float v = in[tp];
                acc[0] = fmaf(v, w0.x, acc[0]); acc[1] = fmaf(v, w0.y, acc[1]);
                acc[2] = fmaf(v, w0.z, acc[2]); acc[3] = fmaf(v, w0.w, acc[3]);
                acc[4] = fmaf(v, w1.x, acc[4]); acc[5] = fmaf(v, w1.y, acc[5]);
                acc[6] = fmaf(v, w1.z, acc[6]); acc[7] = fmaf(v, w1.w, acc[7]);
            }
            if (a.relu) {
#pragma unroll
                for (int j = 0; j < 8; j++) acc[j] = EXT ? act_f(acc[j], a.relu) : fmaxf(acc[j], 0.f);
            }
            uint4 o;
            o.x = pack_bf16(acc[0], acc[1]); o.y = pack_bf16(acc[2], acc[3]);
            o.z = pack_bf16(acc[4], acc[5]); o.w = pack_bf16(acc[6], acc[7]);
            *reinterpret_cast<uint4*>(orow + c8 * 8) = o;
        }
    }
}

__global__ void k_f32_to_bf16(const float* in, __nv_bfloat16* out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = __float2bfloat16_rn(in[i]);
}

__global__ void k_bf16_to_f32(const __nv_bfloat16* in, float* out, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = __bfloat162float(in[i]);
}

// ------------------------------------------------------------------ host side
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

// 2-D bf16 row-major view [rows][cols] with row pitch ld (elements); box = [box_rows][64 cols], 128B swizzle
int make_tmap(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld, uint32_t box_rows) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { pifpaf::set_error("cuTensorMapEncodeTiled entry point not available"); return PIFPAF_E_CUDA; }
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * 2};
    const cuuint32_t box[2] = {BK, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pifpaf::set_error("cuTensorMapEncodeTiled failed (%d): rows=%llu cols=%llu ld=%llu box_rows=%u base=%p",
                          (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld,
                          box_rows, base);
        return PIFPAF_E_CUDA;
    }
    return PIFPAF_OK;
}

// 2-D bf16 row-major view, un-swizzled box [box_rows][box_cols] (dense rows in shared memory)
int make_tmap_plain(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                    uint32_t box_cols, uint32_t box_rows) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { pifpaf::set_error("cuTensorMapEncodeTiled entry point not available"); return PIFPAF_E_CUDA; }
    const cuuint64_t dims[2] = {cols, rows};
    const cuuint64_t strides[1] = {ld * 2};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pifpaf::set_error("cuTensorMapEncodeTiled (plain) failed (%d): rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                          (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
        return PIFPAF_E_CUDA;
    }
    return PIFPAF_OK;
}

// 4-D bf16 NHWC activation view {C, W, H, B} for implicit-GEMM convolutions: box = 64 channels x the
// input window of a PH x PW output patch, traversed with the conv stride
int make_tmap_conv(CUtensorMap* map, const void* base, uint64_t c, uint64_t w, uint64_t h, uint64_t b, uint64_t ld,
                   int stride) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { pifpaf::set_error("cuTensorMapEncodeTiled entry point not available"); return PIFPAF_E_CUDA; }
    const cuuint64_t dims[4] = {c, w, h, b};
    const cuuint64_t strides[3] = {ld * 2, w * ld * 2, h * w * ld * 2};
    const cuuint32_t box[4] = {BK, (cuuint32_t)((PW - 1) * stride + 1), (cuuint32_t)((PH - 1) * stride + 1), 1};
    const cuuint32_t estr[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pifpaf::set_error("cuTensorMapEncodeTiled (conv) failed (%d): c=%llu w=%llu h=%llu b=%llu ld=%llu stride=%d",
                          (int)r, (unsigned long long)c, (unsigned long long)w, (unsigned long long)h,
                          (unsigned long long)b, (unsigned long long)ld, stride);
        return PIFPAF_E_CUDA;
    }
    return PIFPAF_OK;
}

// 4-D bf16 NHWC view {C, W, H, B}, dense (un-swizzled) box of 64 channels x box_w x box_h pixels.
// No L2 promotion: the 128-byte channel block of a pixel is all the kernel wants from that pixel for a long time
// (the channel block is the slowest work index) and pixel strides of 352 / 704 bytes leave most blocks straddling
// 128-byte lines.  ncu (round 1): 256-byte promotion read 2x the algorithmic bytes from DRAM; 128-byte promotion
// requested 1.5x the sectors of no promotion for the same DRAM bytes.
int make_tmap_dw(CUtensorMap* map, const void* base, uint64_t c, uint64_t w, uint64_t h, uint64_t b, uint64_t ld,
                 uint32_t box_w, uint32_t box_h) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { pifpaf::set_error("cuTensorMapEncodeTiled entry point not available"); return PIFPAF_E_CUDA; }
    const cuuint64_t dims[4] = {c, w, h, b};
    const cuuint64_t strides[3] = {ld * 2, w * ld * 2, h * w * ld * 2};
    const cuuint32_t box[4] = {64, box_w, box_h, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pifpaf::set_error("cuTensorMapEncodeTiled (dw) failed (%d): c=%llu w=%llu h=%llu b=%llu ld=%llu box=%ux%u", (int)r,
                          (unsigned long long)c, (unsigned long long)w, (unsigned long long)h, (unsigned long long)b,
                          (unsigned long long)ld, box_w, box_h);
        return PIFPAF_E_CUDA;
    }
    return PIFPAF_OK;
}

// 4-D bf16 NHWC view {C, W, H, B} for the tensor-core depthwise kernel: 64 channels x plane_w x box_h window pixels,
// SWIZZLE_128B (one 128-byte row per pixel: the K-major UMMA A layout), every x_stride-th column (stride 2: one
// column-phase plane per load)
int make_tmap_dw_tc(CUtensorMap* map, const void* base, uint64_t c, uint64_t w, uint64_t h, uint64_t b, uint64_t ld,
                    uint32_t plane_w, uint32_t box_h, uint32_t x_stride) {
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { pifpaf::set_error("cuTensorMapEncodeTiled entry point not available"); return PIFPAF_E_CUDA; }
    const cuuint64_t dims[4] = {c, w, h, b};
    const cuuint64_t strides[3] = {ld * 2, w * ld * 2, h * w * ld * 2};
    const cuuint32_t box[4] = {64, (plane_w - 1) * x_stride + 1, box_h, 1};
    const cuuint32_t estr[4] = {1, x_stride, 1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        pifpaf::set_error("cuTensorMapEncodeTiled (dw tc) failed (%d): c=%llu w=%llu h=%llu b=%llu ld=%llu box=%ux%u stride=%u",
                          (int)r, (unsigned long long)c, (unsigned long long)w, (unsigned long long)h,
                          (unsigned long long)b, (unsigned long long)ld, plane_w, box_h, x_stride);
        return PIFPAF_E_CUDA;
    }
    return PIFPAF_OK;
}

// launch with (or without) the programmatic-stream-serialization attribute
template <typename... KArgs, typename... Args>
cudaError_t launch_kc(bool pdl, int cluster, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                      Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int n = 0;
    if (pdl) {
        attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[n].val.programmaticStreamSerializationAllowed = 1;
        n++;
    }
    if (cluster > 1) {
        attr[n].id = cudaLaunchAttributeClusterDimension;
        attr[n].val.clusterDim.x = (unsigned)cluster; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
        n++;
    }
    cfg.attrs = attr; cfg.numAttrs = n;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
cudaError_t launch_k(bool pdl, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    return launch_kc(pdl, 1, kernel, grid, block, smem, st, std::forward<Args>(args)...);
}

struct Tensor { int h, w, c; __nv_bfloat16* data; };

enum OpKind { OP_INPUT_CONV, OP_GEMM, OP_DW, OP_FUSED, OP_SE };

struct Op {
    OpKind kind;
    // gemm
    GemmArgs g{};
    CUtensorMap tmap_a{}, tmap_b{}, tmap_src{};
    CUtensorMap tmap_bh{}; int pair_resident = 0, pair_stages = 0; size_t pair_smem = 0; bool pair = false;   // k_gemm_tc2
    int a_tensor = -1; int rows_per_image = 0; int tiles_per_image = 0;
    size_t smem = 0;
    // dw
    DwArgs dw{};
    CUtensorMap tmap_dw{}; bool dw_tma = false;
    CUtensorMap tmap_dw_tc{}; bool dw_tc = false;      // tensor-core depthwise (k_dwconv5_tc)
    DwNcArgs dwnc{}; bool dw_nc = false;               // k_dwconv_nc (MobileNet depthwise: k 3 / 5, any activation, SE sums)
    SeArgs se{};                                       // OP_SE (k_se)
    // fused depthwise -> GEMM (OP_FUSED): g + tmap_dw (windows) + tmap_b
    FusedArgs fu{};
    // input conv
    InConvArgs ic{};
    int n_out_pixels = 0;
    double flops_per_image = 0;
    double bytes_per_image = 0;      // algorithmic activation bytes (inputs once + outputs once)
    double weight_bytes = 0;
    int n_real = 0;                  // output channels that are not padding (emit_gemm)
};

}  // namespace

struct pifpaf_net {
    int device = 0, max_batch = 0, n_sm = 148;
    std::vector<Tensor> tensors;
    std::vector<Op> ops;
    std::vector<void*> owned;            // device allocations (weights, biases, tables)
    // heads
    int n_heads = 0;
    // head outputs, optionally double buffered: forward i writes head_out[i & 1] so that a decode of forward i-1
    // (another stream) may still read the other set (pifpaf_net_set_head_buffers)
    float* head_out[2][4] = {{nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr}};
    int head_buffers = 1, head_cur = 0;
    size_t head_elems[4] = {0, 0, 0, 0};
    bool setup_synced = false;           // build-time memsets / uploads (legacy stream) ordered before the first forward
    int sm_limit = 0;                    // > 0: persistent grids use at most this many SMs
    bool pdl = true;                     // programmatic dependent launch between the ops of a forward (PIFPAF_PDL=0: off)
    int gemm_pair = 27;                  // k_gemm_tc2 (CTA pairs, cta_group::2): bit mask of the GEMM classes that use it (PIFPAF_GEMM_PAIR)
    int gemm_debug = 0;                  // GemmArgs::debug for every tcgen05 GEMM launch (PIFPAF_GEMM_DEBUG; timing experiments, wrong results)
    int gemm_mc = 0;                     // weights-resident GEMMs with two n blocks: cluster of two CTAs, A by TMA multicast (PIFPAF_GEMM_MC)
    int gemm_res_stages = 0;             // weights-resident GEMMs: split N further until this many A stages fit (PIFPAF_GEMM_RES_STAGES)
    int dw_tc = 0;                       // depthwise 5x5 on the tensor cores: bit 0 stride 1, bit 1 stride 2 (PIFPAF_DW_TC)
    int dw_tc_pwid = 12, dw_tc_bo = 0;   // descriptor experiments (PIFPAF_DW_TC_PWID = 12 | 16, PIFPAF_DW_TC_BO = 0 | 1)
    bool dw_cbf = false;                 // stride-2 depthwise: channel-block-fastest item order (PIFPAF_DW_CBF=1; measured neutral)
    int head_fields[4] = {0, 0, 0, 0}, head_comp[4] = {0, 0, 0, 0}, head_h = 0, head_w = 0;
    int in_h = 0, in_w = 0;
};

namespace {

template <typename T>
int net_alloc(pifpaf_net* net, T** p, size_t n, bool zero) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), sizeof(T) * (n ? n : 1));
    if (e != cudaSuccess) {
        pifpaf::set_error("cudaMalloc of %zu bytes failed: %s", sizeof(T) * n, cudaGetErrorString(e));
        return e == cudaErrorMemoryAllocation ? PIFPAF_E_NOMEM : PIFPAF_E_CUDA;
    }
    net->owned.push_back(*p);
    net->setup_synced = false;
    if (zero) {
        e = cudaMemset(*p, 0, sizeof(T) * (n ? n : 1));
        if (e != cudaSuccess) { pifpaf::set_error("cudaMemset failed: %s", cudaGetErrorString(e)); return PIFPAF_E_CUDA; }
    }
    return PIFPAF_OK;
}

template <typename T>
int net_upload(pifpaf_net* net, T** p, const std::vector<T>& host) {
    int rc = net_alloc(net, p, host.size(), false);
    if (rc != PIFPAF_OK) return rc;
    cudaError_t e = cudaMemcpy(*p, host.data(), sizeof(T) * host.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { pifpaf::set_error("cudaMemcpy failed: %s", cudaGetErrorString(e)); return PIFPAF_E_CUDA; }
    return PIFPAF_OK;
}

inline int pad8(int v) { return (v + 7) & ~7; }
inline int pad16(int v) { return (v + 15) & ~15; }

// choose the UMMA N tile (<= 256, multiple of 16): the LARGEST tile whose padded work is within
// 10 % of the minimum over all tilings (tiny tiles waste the epilogue and the weight-resident mode; N = 368 must
// become 2 x 192, not 23 x 16)
void choose_block_n(int n_out, int* block_n, int* n_blocks) {
    const int np = pad16(n_out);
    long min_cost = -1;
    for (int nb = 1; nb <= np / 16; nb++) {
        const int bn = pad16((np + nb - 1) / nb);
        if (bn > 256) continue;
        const long cost = (long)bn * nb;
        if (min_cost < 0 || cost < min_cost) min_cost = cost;
    }
    for (int nb = 1; nb <= np / 16; nb++) {
        const int bn = pad16((np + nb - 1) / nb);
        if (bn > 256) continue;
        if ((long)bn * nb * 100 <= min_cost * 110) { *block_n = bn; *n_blocks = nb; return; }
    }
    *block_n = 16; *n_blocks = np / 16;
}

constexpr size_t GEMM_SMEM_BUDGET = 222 * 1024;

size_t gemm_smem_bytes(int block_n, int n_blocks, int stages, bool shuffle, bool b_resident = false, int num_k_blocks = 0) {
    const size_t b_stage = b_resident ? 0 : (size_t)block_n * BK * 2;
    const size_t b_res = b_resident ? (size_t)num_k_blocks * block_n * BK * 2 : 0;
    return 1024 + (size_t)stages * (BM * BK * 2 + b_stage) + b_res + (shuffle ? 2 * (size_t)BM * block_n * 2 : 0) +
           (size_t)n_blocks * block_n * 5 + (2 * stages + 7) * 8 + 64;      // bias (4 B) + scatter table (1 B) per column
}

int choose_stages(int block_n, int n_blocks, int num_k_blocks, bool shuffle) {
    int stages = std::min(8, std::max(2, num_k_blocks * 2));
    while (stages > 2 && gemm_smem_bytes(block_n, n_blocks, stages, shuffle) > GEMM_SMEM_BUDGET) stages--;
    return stages;
}

// weights-resident mode if the whole weight tile plus >= 3 A stages (and the pass-through double buffer) fit
void plan_gemm_smem(GemmArgs& g, size_t* smem, bool src_tma) {
    g.b_resident = 0;
    if (g.conv_k == 0 && g.mode != MODE_HEADS &&
        gemm_smem_bytes(g.block_n, g.n_blocks, 3, src_tma, true, g.num_k_blocks) <= GEMM_SMEM_BUDGET) {
        int stages = 8;
        while (gemm_smem_bytes(g.block_n, g.n_blocks, stages, src_tma, true, g.num_k_blocks) > GEMM_SMEM_BUDGET) stages--;
        g.b_resident = 1;
        g.stages = stages;
        *smem = gemm_smem_bytes(g.block_n, g.n_blocks, stages, src_tma, true, g.num_k_blocks);
        return;
    }
    g.stages = choose_stages(g.block_n, g.n_blocks, g.num_k_blocks, src_tma);
    *smem = gemm_smem_bytes(g.block_n, g.n_blocks, g.stages, src_tma);
}

// multicast pairs (GemmArgs::mc): weights-resident GEMMs whose N takes two n blocks read every A tile twice, once per
// n block, and the second read is what bounds them (profiles/r2_history.md, session l: 43 us per pass over A)
int plan_gemm_mc(pifpaf_net* net, Op& op, const Tensor& tin) {
    GemmArgs& g = op.g;
    g.mc = 0;
    if (!net->gemm_mc || !g.b_resident || g.n_blocks != 2 || g.src_tma || g.conv_k != 0) return PIFPAF_OK;
    if (g.mode != MODE_PLAIN && g.mode != MODE_SCATTER) return PIFPAF_OK;
    g.mc = 1;
    return make_tmap(&op.tmap_src, tin.data, (uint64_t)net->max_batch * tin.h * tin.w, (uint64_t)tin.c, (uint64_t)tin.c, BM / 2);
}

// CTA pairs (k_gemm_tc2): each CTA stages half of the weight tile.  PIFPAF_GEMM_PAIR is a mask of GEMM classes:
//   1  weights-resident, two or more n blocks (stage 3: 0.150 -> 0.130 ms per launch, session o)
//   2  streaming (stage 4, conv5, the 1x1 in front of a stride-2 depthwise: 0.109 -> 0.091, 0.377 -> 0.330)
//   4  weights-resident, one n block, several K blocks (stage 2: DRAM-bound already, 0.208 -> 0.235: off)
//   8  weights-resident, one n block, one K block (the K = 32 GEMM at 321 x 321: 0.602 -> 0.544)
//  16  the heads GEMM
int plan_gemm_pair(pifpaf_net* net, Op& op) {
    GemmArgs& g = op.g;
    op.pair = false;
    if (!net->gemm_pair || g.src_tma || g.conv_k != 0 || g.mc) return PIFPAF_OK;
    if (g.mode != MODE_PLAIN && g.mode != MODE_SCATTER && g.mode != MODE_HEADS) return PIFPAF_OK;
    const int want = g.mode == MODE_HEADS ? 16 : g.b_resident ? (g.n_blocks >= 2 ? 1 : (g.num_k_blocks <= 1 ? 8 : 4)) : 2;
    if (!(net->gemm_pair & want)) return PIFPAF_OK;
    const size_t n_pad = (size_t)g.block_n * g.n_blocks;
    const size_t bh = (size_t)(g.block_n / 2) * BK * 2;
    const size_t fixed = 1024 + n_pad * 4 + n_pad / 16 * sizeof(DestGroup) + 64;
    auto total = [&](int stages, bool res) {
        const size_t b_res = res ? (((size_t)g.num_k_blocks * bh + 1023) & ~(size_t)1023) : 0;
        return fixed + (size_t)stages * (BM * BK * 2 + (res ? 0 : bh)) + b_res + (2 * (size_t)stages + 5) * 8;
    };
    const bool res = g.mode != MODE_HEADS && total(4, true) <= GEMM_SMEM_BUDGET;
    int stages = PAIR_MAX_STAGES;
    while (stages > 2 && total(stages, res) > GEMM_SMEM_BUDGET) stages--;
    op.pair = true; op.pair_resident = res ? 1 : 0; op.pair_stages = stages; op.pair_smem = total(stages, res);
    return make_tmap(&op.tmap_bh, g.wgt, (uint64_t)n_pad, (uint64_t)g.ldw, (uint64_t)g.ldw, (uint32_t)(g.block_n / 2));
}

// common GEMM emit: weights [n_out][k_cols] f32 host -> bf16 [n_pad][k_pad8] device, bias padded
int emit_gemm(pifpaf_net* net, Op& op, int in_tensor, int in_col_off, int k_cols, int n_out,
              const float* weight, const float* bias) {
    const Tensor& tin = net->tensors[in_tensor];
    // measured on B200: a TMA inner coordinate that is not 16-byte aligned raises an illegal-instruction fault
    PIFPAF_CHECK_ARG(in_col_off >= 0 && in_col_off % 8 == 0 && in_col_off + k_cols <= tin.c,
                     "conv1x1 input column window must start on a multiple of 8 channels and lie inside the tensor");
    int block_n, n_blocks;
    choose_block_n(n_out, &block_n, &n_blocks);
    // weights-resident GEMMs stream A through what the resident weight tile leaves of the shared memory: with
    // K = 352..416 and a 176..208-column tile that is 4-5 stages of 16 KB, too few bytes in flight per SM to cover
    // the DRAM latency (the K <= 208 launches with 8 stages reach 5.5-6 TB/s, these 3.4-4.2).  Narrower tiles (more
    // n blocks, A re-read from L2 by each of them) buy the stages back.
    if (net->gemm_res_stages > 0) {
        const int kb = (k_cols + BK - 1) / BK, np = pad16(n_out);
        auto res_stages = [&](int bn, int nb) {
            if (gemm_smem_bytes(bn, nb, 3, false, true, kb) > GEMM_SMEM_BUDGET) return 0;       // not resident at all
            int st = 8;
            while (gemm_smem_bytes(bn, nb, st, false, true, kb) > GEMM_SMEM_BUDGET) st--;
            return st;
        };
        int st = res_stages(block_n, n_blocks);
        while (st > 0 && st < net->gemm_res_stages && block_n > 64) {
            const int nb = n_blocks + 1, bn = pad16((np + nb - 1) / nb);
            if (bn < 64) break;
            n_blocks = nb; block_n = bn;
            st = res_stages(block_n, n_blocks);
        }
    }
    const int n_pad = block_n * n_blocks;
    const int k_pad = pad8(k_cols);
    std::vector<__nv_bfloat16> w((size_t)n_pad * k_pad, __float2bfloat16(0.f));
    for (int n = 0; n < n_out; n++)
        for (int k = 0; k < k_cols; k++) w[(size_t)n * k_pad + k] = __float2bfloat16(weight[(size_t)n * k_cols + k]);
    std::vector<float> b(n_pad, 0.f);
    for (int n = 0; n < n_out; n++) b[n] = bias ? bias[n] : 0.f;
    __nv_bfloat16* d_w = nullptr; float* d_b = nullptr;
    int rc = net_upload(net, &d_w, w); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b, b); if (rc != PIFPAF_OK) return rc;

    GemmArgs& g = op.g;
    const size_t rows_max = (size_t)net->max_batch * tin.h * tin.w;
    g.N = n_out; g.K = k_cols; g.a_col0 = in_col_off;
    g.block_n = block_n; g.n_blocks = n_blocks;
    g.num_k_blocks = (k_cols + BK - 1) / BK;
    g.stages = choose_stages(block_n, n_blocks, g.num_k_blocks, false);
    g.bias = d_b;
    g.a = tin.data + in_col_off; g.lda = tin.c; g.wgt = d_w; g.ldw = k_pad;
    op.a_tensor = in_tensor; op.rows_per_image = tin.h * tin.w;
    op.smem = gemm_smem_bytes(block_n, n_blocks, g.stages, false);
    // ALGORITHMIC work: padding columns / rows (zero weights: view lead-ins of the 'shuffle' layout, 16-channel
    // padding of the 'bins' pieces) are not counted -- nnz MACs, the input channels some weight reads, the output
    // channels some weight or bias produces
    long long nnz = 0; int k_real = 0, n_real = 0;
    {
        std::vector<char> k_used(k_cols, 0);
        for (int n = 0; n < n_out; n++) {
            bool row = bias != nullptr && bias[n] != 0.f;
            for (int k = 0; k < k_cols; k++)
                if (weight[(size_t)n * k_cols + k] != 0.f) { nnz++; k_used[k] = 1; row = true; }
            n_real += row ? 1 : 0;
        }
        for (int k = 0; k < k_cols; k++) k_real += k_used[k];
    }
    op.n_real = n_real;
    op.flops_per_image = 2.0 * (double)op.rows_per_image * (double)nnz;
    op.bytes_per_image = (double)op.rows_per_image * k_real * 2.0;      // A read once (bf16); outputs added by the caller
    op.weight_bytes = (double)nnz * 2.0;
    // the map covers the whole tensor; the view's first column is a TMA coordinate (16-byte aligned).
    // Columns past the view multiply zero weight rows (B is zero padded), columns past the tensor are zero filled.
    rc = make_tmap(&op.tmap_a, tin.data, rows_max, (uint64_t)tin.c, (uint64_t)tin.c, BM);
    if (rc != PIFPAF_OK) return rc;
    rc = make_tmap(&op.tmap_b, d_w, (uint64_t)n_pad, (uint64_t)k_pad, (uint64_t)k_pad, (uint32_t)block_n);
    return rc;
}

// k_dwconv_nc work split: CTA = blockDim * nit items of one image, blockDim a multiple of C8 (so a thread keeps its
// channel group); nit from the image size alone, so that the squeeze-excitation sum slots do not depend on the batch
void plan_dw_nc(const DwArgs& a, DwNcArgs* x, int* block) {
    const int bd = (256 / a.C8) * a.C8;
    const int per_img = a.Hout * ((a.Wout + DW_OX - 1) / DW_OX) * a.C8;
    x->nit = std::max(1, std::min(16, per_img / (bd * 16)));
    x->nslots = (per_img + bd * x->nit - 1) / (bd * x->nit);
    *block = bd;
}

// dense kxk conv as an implicit GEMM on tensor cores (8 x 16 output-pixel patches of one image per M tile).
// wproj_f32 != nullptr: per-image weights (squeeze-excitation projection, kernel 1): B holds max_batch copies of the
// weight matrix, written by k_se; *wproj_f32 receives the f32 weights [n_pad][k_total] k_se scales.
int emit_conv_gemm(pifpaf_net* net, Op& op, int in_tensor, int in_col_off, int c_in, int kernel, int stride, int pad,
                   int n_out, const float* weight, const float* bias, int relu, int out_tensor, int out_col_off,
                   int residual_tensor, int residual_col_off, float** wproj_f32) {
    const int nt = (int)net->tensors.size();
    const Tensor& tin = net->tensors[in_tensor];
    const Tensor& to = net->tensors[out_tensor];
    const int ho = (tin.h + 2 * pad - kernel) / stride + 1, wo = (tin.w + 2 * pad - kernel) / stride + 1;
    int block_n, n_blocks;
    choose_block_n(n_out, &block_n, &n_blocks);
    const int n_pad = block_n * n_blocks;
    const int taps = kernel * kernel, cblocks = (c_in + BK - 1) / BK;
    const int k_total = taps * cblocks * BK;
    // torch weight [n_out][c_in][k][k] -> bf16 [n_pad][tap][cblocks*64]
    std::vector<__nv_bfloat16> w((size_t)n_pad * k_total, __float2bfloat16(0.f));
    for (int n = 0; n < n_out; n++)
        for (int c = 0; c < c_in; c++)
            for (int t = 0; t < taps; t++)
                w[(size_t)n * k_total + (size_t)t * cblocks * BK + c] = __float2bfloat16(weight[((size_t)n * c_in + c) * taps + t]);
    std::vector<float> b(n_pad, 0.f);
    for (int n = 0; n < n_out; n++) b[n] = bias ? bias[n] : 0.f;
    __nv_bfloat16* d_w = nullptr; float* d_b = nullptr;
    int rc = net_upload(net, &d_b, b); if (rc != PIFPAF_OK) return rc;
    uint64_t b_rows = (uint64_t)n_pad;
    if (wproj_f32 == nullptr) {
        rc = net_upload(net, &d_w, w); if (rc != PIFPAF_OK) return rc;
    } else {
        // per-image weights: k_se writes image b's copy of the weights into rows [b * n_pad, (b + 1) * n_pad)
        PIFPAF_CHECK_ARG(kernel == 1, "per-image weights need kernel 1");
        std::vector<float> wf(w.size(), 0.f);
        for (int n = 0; n < n_out; n++)
            for (int c = 0; c < c_in; c++) wf[(size_t)n * k_total + c] = weight[(size_t)n * c_in + c];
        float* d_wf = nullptr;
        rc = net_upload(net, &d_wf, wf); if (rc != PIFPAF_OK) return rc;
        *wproj_f32 = d_wf;
        b_rows = (uint64_t)net->max_batch * n_pad;
        rc = net_alloc(net, &d_w, (size_t)b_rows * k_total, true); if (rc != PIFPAF_OK) return rc;
        op.g.w_img_rows = n_pad;
    }
    GemmArgs& g = op.g;
    g.N = n_out; g.K = c_in;
    g.block_n = block_n; g.n_blocks = n_blocks;
    g.num_k_blocks = taps * cblocks;
    g.stages = choose_stages(block_n, n_blocks, g.num_k_blocks, false);
    g.bias = d_b; g.mode = MODE_PLAIN; g.relu = relu;
    g.out = to.data; g.ldo = to.c; g.out_col_off = out_col_off;
    g.conv_k = kernel; g.conv_stride = stride; g.conv_pad = pad; g.conv_cblocks = cblocks;
    g.Hi = tin.h; g.Wi = tin.w; g.Ho = ho; g.Wo = wo;
    g.tiles_x = (wo + PW - 1) / PW; g.tiles_y = (ho + PH - 1) / PH;
    g.a = tin.data + in_col_off; g.lda = tin.c; g.wgt = d_w; g.ldw = k_total;
    if (residual_tensor >= 0) {
        PIFPAF_CHECK_ARG(residual_tensor < nt, "bad residual tensor");
        const Tensor& tr = net->tensors[residual_tensor];
        PIFPAF_CHECK_ARG(tr.h == ho && tr.w == wo && residual_col_off % 8 == 0 && residual_col_off + n_out <= tr.c,
                         "residual tensor shape mismatch");
        g.res = tr.data; g.ld_res = tr.c; g.res_col_off = residual_col_off;
    }
    op.a_tensor = in_tensor; op.rows_per_image = ho * wo; op.tiles_per_image = g.tiles_x * g.tiles_y;
    op.smem = gemm_smem_bytes(block_n, n_blocks, g.stages, false);
    op.flops_per_image = 2.0 * (double)ho * wo * n_out * c_in * taps;
    op.bytes_per_image = (double)tin.h * tin.w * c_in * 2.0 + (double)ho * wo * n_out * 2.0 * (residual_tensor >= 0 ? 2.0 : 1.0);
    op.weight_bytes = (double)n_out * c_in * taps * 2.0;
    rc = make_tmap_conv(&op.tmap_a, tin.data + in_col_off, (uint64_t)c_in, (uint64_t)tin.w, (uint64_t)tin.h,
                        (uint64_t)net->max_batch, (uint64_t)tin.c, stride);
    if (rc != PIFPAF_OK) return rc;
    return make_tmap(&op.tmap_b, d_w, b_rows, (uint64_t)k_total, (uint64_t)k_total, (uint32_t)block_n);
}

}  // namespace

extern "C" {

int pifpaf_net_create(pifpaf_net_t** out, int32_t device, int32_t max_batch) {
    PIFPAF_CHECK_ARG(out != nullptr, "out is null");
    *out = nullptr;
    PIFPAF_CHECK_ARG(max_batch >= 1, "max_batch must be >= 1");
    int n_dev = 0;
    PIFPAF_CUDA_TRY(cudaGetDeviceCount(&n_dev));
    PIFPAF_CHECK_ARG(device >= 0 && device < n_dev, "no such CUDA device");
    PIFPAF_CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    PIFPAF_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        pifpaf::set_error("libpifpaf_b200 is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
        return PIFPAF_E_CUDA;
    }
    pifpaf_net* net = new pifpaf_net();
    net->device = device; net->max_batch = max_batch; net->n_sm = prop.multiProcessorCount;
    if (const char* e = std::getenv("PIFPAF_DW_CBF")) net->dw_cbf = std::atoi(e) != 0;
    if (const char* e = std::getenv("PIFPAF_PDL")) net->pdl = std::atoi(e) != 0;
    if (const char* e = std::getenv("PIFPAF_GEMM_RES_STAGES")) net->gemm_res_stages = std::atoi(e);
    if (const char* e = std::getenv("PIFPAF_GEMM_MC")) net->gemm_mc = std::atoi(e);
    if (const char* e = std::getenv("PIFPAF_GEMM_DEBUG")) net->gemm_debug = std::atoi(e);
    if (const char* e = std::getenv("PIFPAF_GEMM_PAIR")) net->gemm_pair = std::atoi(e);
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_gemm_tc2<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_gemm_tc2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    if (const char* e = std::getenv("PIFPAF_DW_TC")) net->dw_tc = std::atoi(e);
    if (const char* e = std::getenv("PIFPAF_DW_TC_PWID")) net->dw_tc_pwid = std::atoi(e) == 16 ? 16 : 12;
    if (const char* e = std::getenv("PIFPAF_DW_TC_BO")) net->dw_tc_bo = std::atoi(e) != 0;
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dwconv5_tc<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dwconv5_tc<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_gemm_tc<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_gemm_tc<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dwconv5_tma<1, DW1_TH, DW1_TW, 4, 3>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, DwS1::SMEM));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dwconv5_tma<2, DW2_TH, DW2_TW, 4, 2>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, DwS2::SMEM));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dwconv5_tma<2, DW2_TH, DW2_TW, 4, 2, true>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    PIFPAF_CUDA_TRY(cudaFuncSetAttribute(k_dw_gemm<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    *out = net;
    return PIFPAF_OK;
}

void pifpaf_net_destroy(pifpaf_net_t* net) {
    if (!net) return;
    cudaSetDevice(net->device);
    for (void* p : net->owned) cudaFree(p);
    delete net;
}

int pifpaf_net_tensor(pifpaf_net_t* net, int32_t h, int32_t w, int32_t c_phys, int32_t* id) {
    PIFPAF_CHECK_ARG(net != nullptr && id != nullptr, "null argument");
    PIFPAF_CHECK_ARG(h >= 1 && w >= 1 && c_phys >= 16 && c_phys % 16 == 0, "tensor shape: c_phys must be a multiple of 16");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    Tensor t; t.h = h; t.w = w; t.c = c_phys; t.data = nullptr;
    // + one tile of slack rows so that TMA boxes of the last partial M tile stay in mapped memory
    int rc = net_alloc(net, &t.data, ((size_t)net->max_batch * h * w + BM) * c_phys, true);
    if (rc != PIFPAF_OK) return rc;
    net->tensors.push_back(t);
    *id = (int)net->tensors.size() - 1;
    return PIFPAF_OK;
}

int pifpaf_net_input_conv(pifpaf_net_t* net, int32_t in_h, int32_t in_w, int32_t kernel, int32_t stride,
                          int32_t pad, int32_t c_out, const float* weight, const float* bias,
                          int32_t relu, int32_t out_tensor) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr, "null argument");
    PIFPAF_CHECK_ARG(relu >= 0 && relu <= 3, "activation code must be 0..3");
    PIFPAF_CHECK_ARG(out_tensor >= 0 && out_tensor < (int)net->tensors.size(), "bad tensor id");
    const Tensor& to = net->tensors[out_tensor];
    const int ho = (in_h + 2 * pad - kernel) / stride + 1, wo = (in_w + 2 * pad - kernel) / stride + 1;
    PIFPAF_CHECK_ARG(to.h == ho && to.w == wo && to.c >= pad8(c_out), "output tensor shape mismatch");
    PIFPAF_CHECK_ARG(kernel == 1 || kernel == 3 || kernel == 5 || kernel == 7, "input conv kernel must be 1, 3, 5 or 7");
    PIFPAF_CHECK_ARG(relu <= 1 || kernel == 3, "activation codes 2 and 3 need a 3x3 input conv");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    const int C = pad8(c_out);
    std::vector<float> w((size_t)3 * kernel * kernel * C, 0.f), b(C, 0.f);
    for (int co = 0; co < c_out; co++) {
        for (int ci = 0; ci < 3; ci++)
            for (int ky = 0; ky < kernel; ky++)
                for (int kx = 0; kx < kernel; kx++)
                    w[(size_t)((ci * kernel + ky) * kernel + kx) * C + co] =
                        weight[(((size_t)co * 3 + ci) * kernel + ky) * kernel + kx];
        b[co] = bias ? bias[co] : 0.f;
    }
    Op op; op.kind = OP_INPUT_CONV;
    float *d_w = nullptr, *d_b = nullptr;
    int rc = net_upload(net, &d_w, w); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b, b); if (rc != PIFPAF_OK) return rc;
    InConvArgs& a = op.ic;
    a.in = nullptr; a.out = to.data; a.ld_out = to.c; a.weight = d_w; a.bias = d_b;
    a.Hin = in_h; a.Win = in_w; a.Hout = ho; a.Wout = wo; a.C8 = C / 8;
    a.kernel = kernel; a.stride = stride; a.pad = pad; a.relu = relu;
    op.flops_per_image = 2.0 * ho * wo * c_out * 3.0 * kernel * kernel;
    op.bytes_per_image = (double)in_h * in_w * 3 * 4.0 + (double)ho * wo * c_out * 2.0;
    net->in_h = in_h; net->in_w = in_w;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_conv1x1(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t k_cols,
                       int32_t n_out, const float* weight, const float* bias, int32_t relu,
                       int32_t out_tensor, int32_t out_col_off,
                       int32_t shuffle_src_tensor, int32_t shuffle_src_col_off) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr, "null argument");
    PIFPAF_CHECK_ARG(relu >= 0 && relu <= 3, "activation code must be 0..3");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt && out_tensor >= 0 && out_tensor < nt, "bad tensor id");
    PIFPAF_CHECK_ARG(k_cols >= 1 && n_out >= 1, "bad conv size");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    const Tensor& tin = net->tensors[in_tensor];
    const Tensor& to = net->tensors[out_tensor];
    PIFPAF_CHECK_ARG(tin.h == to.h && tin.w == to.w, "conv1x1 keeps the spatial shape");
    Op op; op.kind = OP_GEMM;
    int rc = emit_gemm(net, op, in_tensor, in_col_off, k_cols, n_out, weight, bias);
    if (rc != PIFPAF_OK) return rc;
    GemmArgs& g = op.g;
    g.relu = relu; g.out = to.data; g.ldo = to.c; g.out_col_off = out_col_off;
    // outputs: n_out bf16 per row; the fused shuffle also reads and re-writes the pass-through half
    op.bytes_per_image += (double)op.rows_per_image * op.n_real * 2.0 * (shuffle_src_tensor >= 0 ? 3.0 : 1.0);
    PIFPAF_CHECK_ARG(out_col_off % 16 == 0, "output column offset must be a multiple of 16");
    if (shuffle_src_tensor < 0) {
        g.mode = MODE_PLAIN;
        PIFPAF_CHECK_ARG(out_col_off + pad8(n_out) <= to.c, "output window outside the tensor");
    } else {
        PIFPAF_CHECK_ARG(shuffle_src_tensor < nt, "bad shuffle source tensor");
        const Tensor& ts = net->tensors[shuffle_src_tensor];
        PIFPAF_CHECK_ARG(ts.h == to.h && ts.w == to.w, "shuffle source shape mismatch");
        PIFPAF_CHECK_ARG(n_out % 2 == 0, "fused channel_shuffle needs an even branch width");
        PIFPAF_CHECK_ARG(shuffle_src_col_off % 8 == 0 && shuffle_src_col_off + pad16(n_out) <= ts.c + 8,
                         "shuffle source window");
        PIFPAF_CHECK_ARG(out_col_off == 0 && to.c >= 2 * n_out, "shuffle output tensor must hold 2*n_out channels");
        g.mode = MODE_SHUFFLE;
        g.src0 = ts.data; g.ld0 = ts.c; g.src0_col_off = shuffle_src_col_off;
        g.half = n_out; g.gap = 0;
        g.src_tma = gemm_smem_bytes(g.block_n, g.n_blocks, 2, true) <= GEMM_SMEM_BUDGET ? 1 : 0;
        // pass-through tile [BM rows][block_n cols], dense rows in shared memory (no swizzle)
        rc = make_tmap_plain(&op.tmap_src, ts.data + shuffle_src_col_off, (uint64_t)net->max_batch * ts.h * ts.w,
                             (uint64_t)std::min(ts.c - shuffle_src_col_off, pad16(n_out)), (uint64_t)ts.c,
                             (uint32_t)g.block_n, BM);
        if (rc != PIFPAF_OK) return rc;
    }
    plan_gemm_smem(g, &op.smem, g.src_tma != 0);
    rc = plan_gemm_mc(net, op, tin); if (rc != PIFPAF_OK) return rc;
    rc = plan_gemm_pair(net, op); if (rc != PIFPAF_OK) return rc;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_conv1x1_scatter(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t k_cols,
                               int32_t n_out, const float* weight, const float* bias, int32_t relu,
                               int32_t n_pieces, const int32_t* piece_col0, const int32_t* piece_count,
                               const int32_t* piece_tensor, const int32_t* piece_tensor_col) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr && piece_col0 && piece_count && piece_tensor && piece_tensor_col,
                     "null argument");
    PIFPAF_CHECK_ARG(relu >= 0 && relu <= 3, "activation code must be 0..3");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt, "bad tensor id");
    PIFPAF_CHECK_ARG(k_cols >= 1 && n_out >= 16 && n_out % 16 == 0 && n_pieces >= 1, "bad conv size");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    const Tensor& tin = net->tensors[in_tensor];
    Op op; op.kind = OP_GEMM;
    int rc = emit_gemm(net, op, in_tensor, in_col_off, k_cols, n_out, weight, bias);
    if (rc != PIFPAF_OK) return rc;
    GemmArgs& g = op.g;
    g.mode = MODE_SCATTER; g.relu = relu;
    std::vector<DestGroup> groups((size_t)g.n_blocks * g.block_n / 16, DestGroup{nullptr, 0, 0});
    int expect = 0;
    for (int i = 0; i < n_pieces; i++) {
        PIFPAF_CHECK_ARG(piece_col0[i] == expect && piece_count[i] >= 16 && piece_count[i] % 16 == 0,
                         "pieces must tile [0, n_out) in order, in multiples of 16 columns");
        PIFPAF_CHECK_ARG(piece_tensor[i] >= 0 && piece_tensor[i] < nt, "bad piece tensor id");
        const Tensor& to = net->tensors[piece_tensor[i]];
        PIFPAF_CHECK_ARG(to.h == tin.h && to.w == tin.w, "conv1x1 keeps the spatial shape");
        PIFPAF_CHECK_ARG(piece_tensor_col[i] >= 0 && piece_tensor_col[i] % 16 == 0 &&
                         piece_tensor_col[i] + piece_count[i] <= to.c, "piece window outside its tensor");
        for (int c = 0; c < piece_count[i]; c += 16)
            groups[(size_t)(expect + c) / 16] = DestGroup{to.data + piece_tensor_col[i] + c, to.c, 0};
        expect += piece_count[i];
    }
    PIFPAF_CHECK_ARG(expect == n_out, "pieces must cover all n_out columns");
    DestGroup* d_groups = nullptr;
    rc = net_upload(net, &d_groups, groups);
    if (rc != PIFPAF_OK) return rc;
    g.dest = d_groups;
    op.bytes_per_image += (double)op.rows_per_image * op.n_real * 2.0;
    plan_gemm_smem(g, &op.smem, false);
    rc = plan_gemm_mc(net, op, tin); if (rc != PIFPAF_OK) return rc;
    rc = plan_gemm_pair(net, op); if (rc != PIFPAF_OK) return rc;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_conv(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t c_in,
                    int32_t kernel, int32_t stride, int32_t pad, int32_t n_out, const float* weight,
                    const float* bias, int32_t relu, int32_t out_tensor, int32_t out_col_off,
                    int32_t residual_tensor, int32_t residual_col_off) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr, "null argument");
    PIFPAF_CHECK_ARG(relu >= 0 && relu <= 3, "activation code must be 0..3");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt && out_tensor >= 0 && out_tensor < nt, "bad tensor id");
    PIFPAF_CHECK_ARG(kernel >= 1 && kernel <= 7 && stride >= 1 && stride <= 2 && pad >= 0, "unsupported conv geometry");
    PIFPAF_CHECK_ARG(c_in >= 1 && n_out >= 1, "bad conv size");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    const Tensor& tin = net->tensors[in_tensor];
    const Tensor& to = net->tensors[out_tensor];
    const int ho = (tin.h + 2 * pad - kernel) / stride + 1, wo = (tin.w + 2 * pad - kernel) / stride + 1;
    PIFPAF_CHECK_ARG(to.h == ho && to.w == wo, "conv output tensor shape mismatch");
    PIFPAF_CHECK_ARG(in_col_off % 8 == 0 && in_col_off + c_in <= tin.c, "conv input column window");
    PIFPAF_CHECK_ARG(out_col_off % 16 == 0 && out_col_off + pad8(n_out) <= to.c, "conv output column window");
    if (kernel == 1 && stride == 1 && pad == 0) {
        // pointwise: the flat [pixels x channels] GEMM (no patch tiling waste), residual fused the same way
        Op op; op.kind = OP_GEMM;
        int rc = emit_gemm(net, op, in_tensor, in_col_off, c_in, n_out, weight, bias);
        if (rc != PIFPAF_OK) return rc;
        GemmArgs& g = op.g;
        g.mode = MODE_PLAIN; g.relu = relu; g.out = to.data; g.ldo = to.c; g.out_col_off = out_col_off;
        op.bytes_per_image += (double)op.rows_per_image * op.n_real * 2.0 * (residual_tensor >= 0 ? 2.0 : 1.0);
        if (residual_tensor >= 0) {
            PIFPAF_CHECK_ARG(residual_tensor < nt, "bad residual tensor");
            const Tensor& tr = net->tensors[residual_tensor];
            PIFPAF_CHECK_ARG(tr.h == ho && tr.w == wo && residual_col_off % 8 == 0 && residual_col_off + n_out <= tr.c,
                             "residual tensor shape mismatch");
            g.res = tr.data; g.ld_res = tr.c; g.res_col_off = residual_col_off;
        }
        plan_gemm_smem(g, &op.smem, false);
        rc = plan_gemm_mc(net, op, tin); if (rc != PIFPAF_OK) return rc;
        rc = plan_gemm_pair(net, op); if (rc != PIFPAF_OK) return rc;
        net->ops.push_back(op);
        return PIFPAF_OK;
    }
    Op op; op.kind = OP_GEMM;
    int rc = emit_conv_gemm(net, op, in_tensor, in_col_off, c_in, kernel, stride, pad, n_out, weight, bias, relu,
                            out_tensor, out_col_off, residual_tensor, residual_col_off, nullptr);
    if (rc != PIFPAF_OK) return rc;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_dwconv(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t channels,
                      int32_t kernel, int32_t stride, int32_t pad, const float* weight, const float* bias,
                      int32_t relu, int32_t out_tensor, int32_t out_col_off) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr, "null argument");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt && out_tensor >= 0 && out_tensor < nt, "bad tensor id");
    const Tensor& tin = net->tensors[in_tensor];
    const Tensor& to = net->tensors[out_tensor];
    const int ho = (tin.h + 2 * pad - kernel) / stride + 1, wo = (tin.w + 2 * pad - kernel) / stride + 1;
    const int C = pad8(channels);
    PIFPAF_CHECK_ARG(to.h == ho && to.w == wo, "dwconv output tensor shape mismatch");
    PIFPAF_CHECK_ARG(in_col_off % 8 == 0 && out_col_off % 8 == 0 && in_col_off + C <= tin.c && out_col_off + C <= to.c,
                     "dwconv column windows");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    std::vector<float> w((size_t)kernel * kernel * C, 0.f), b(C, 0.f);
    for (int c = 0; c < channels; c++) {
        for (int t = 0; t < kernel * kernel; t++) w[(size_t)t * C + c] = weight[(size_t)c * kernel * kernel + t];
        b[c] = bias ? bias[c] : 0.f;
    }
    Op op; op.kind = OP_DW;
    float *d_w = nullptr, *d_b = nullptr;
    int rc = net_upload(net, &d_w, w); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b, b); if (rc != PIFPAF_OK) return rc;
    DwArgs& a = op.dw;
    a.in = tin.data; a.ld_in = tin.c; a.in_col_off = in_col_off;
    a.out = to.data; a.ld_out = to.c; a.out_col_off = out_col_off;
    a.weight = d_w; a.bias = d_b;
    a.Hin = tin.h; a.Win = tin.w; a.Hout = ho; a.Wout = wo; a.C8 = C / 8;
    a.kernel = kernel; a.stride = stride; a.pad = pad; a.relu = relu;
    op.flops_per_image = 2.0 * ho * wo * channels * (double)kernel * kernel;
    op.bytes_per_image = ((double)tin.h * tin.w + (double)ho * wo) * channels * 2.0;
    const bool nc_geometry = (kernel == 3 || kernel == 5) && (stride == 1 || stride == 2);
    PIFPAF_CHECK_ARG(relu >= 0 && relu <= 3, "activation code must be 0..3");
    PIFPAF_CHECK_ARG(relu <= 1 || nc_geometry, "activation codes 2 and 3 need a 3x3 or 5x5 depthwise conv of stride 1 or 2");
    if (nc_geometry && (kernel == 3 || relu >= 2)) {
        // MobileNet depthwise convs: k_dwconv_nc (5x5 with ReLU or none stays on the TMA kernels below unless a
        // squeeze-excitation follows, pifpaf_net_se_conv1x1)
        PIFPAF_CHECK_ARG(C / 8 <= 256, "depthwise conv of more than 2048 channels");
        op.dw_nc = true;
    } else if (kernel == 5 && (stride == 1 || stride == 2)) {
        const uint32_t bw = stride == 1 ? DwS1::IW : DwS2::IW;
        const uint32_t bh = stride == 1 ? DwS1::IH : DwS2::IH;
        rc = make_tmap_dw(&op.tmap_dw, tin.data + in_col_off, (uint64_t)C, (uint64_t)tin.w, (uint64_t)tin.h,
                          (uint64_t)net->max_batch, (uint64_t)tin.c, bw, bh);
        if (rc != PIFPAF_OK) return rc;
        op.dw_tma = true;
        if (pad == 2 && ((net->dw_tc >> (stride - 1)) & 1)) {
            const uint32_t pw = stride == 1 ? (uint32_t)net->dw_tc_pwid : (uint32_t)DwTc<2>::PWID;
            rc = make_tmap_dw_tc(&op.tmap_dw_tc, tin.data + in_col_off, (uint64_t)C, (uint64_t)tin.w, (uint64_t)tin.h,
                                 (uint64_t)net->max_batch, (uint64_t)tin.c, pw,
                                 stride == 1 ? DwTc<1>::IH : DwTc<2>::IH, (uint32_t)stride);
            if (rc != PIFPAF_OK) return rc;
            op.dw_tc = true;
        }
    }
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_se_conv1x1(pifpaf_net_t* net, int32_t in_tensor, int32_t channels, int32_t squeeze,
                          const float* fc1_weight, const float* fc1_bias, const float* fc2_weight, const float* fc2_bias,
                          int32_t n_out, const float* weight, const float* bias, int32_t out_tensor,
                          int32_t residual_tensor) {
    PIFPAF_CHECK_ARG(net != nullptr && fc1_weight && fc1_bias && fc2_weight && fc2_bias && weight, "null argument");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt && out_tensor >= 0 && out_tensor < nt && residual_tensor < nt,
                     "bad tensor id");
    PIFPAF_CHECK_ARG(channels >= 1 && channels <= 2048 && squeeze >= 1 && squeeze <= 2048 && n_out >= 1, "bad SE size");
    const Tensor& tin = net->tensors[in_tensor];
    const Tensor& to = net->tensors[out_tensor];
    PIFPAF_CHECK_ARG(tin.h == to.h && tin.w == to.w, "the projection keeps the spatial shape");
    PIFPAF_CHECK_ARG(!net->ops.empty() && net->ops.back().kind == OP_DW, "squeeze-excitation must follow a depthwise conv");
    {
        const DwArgs& d = net->ops.back().dw;
        PIFPAF_CHECK_ARG(d.out == tin.data && d.out_col_off == 0 && d.C8 * 8 == pad8(channels),
                         "squeeze-excitation input must be the whole output of the preceding depthwise conv");
        PIFPAF_CHECK_ARG((d.kernel == 3 || d.kernel == 5) && (d.stride == 1 || d.stride == 2),
                         "squeeze-excitation needs a 3x3 or 5x5 depthwise conv of stride 1 or 2");
    }
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    DwNcArgs nc{}; int block = 0;
    plan_dw_nc(net->ops.back().dw, &nc, &block);
    const int C = pad8(channels);
    float* d_part = nullptr;
    int rc = net_alloc(net, &d_part, (size_t)net->max_batch * nc.nslots * C, true); if (rc != PIFPAF_OK) return rc;
    nc.se_part = d_part;
    {
        Op& dw = net->ops.back();
        dw.dw_nc = true;
        dw.dwnc = nc;
        dw.bytes_per_image += (double)nc.nslots * C * 4.0;
    }
    Op gop; gop.kind = OP_GEMM;
    float* d_wproj = nullptr;
    rc = emit_conv_gemm(net, gop, in_tensor, 0, channels, 1, 1, 0, n_out, weight, bias, 0, out_tensor, 0,
                        residual_tensor, 0, &d_wproj);
    if (rc != PIFPAF_OK) return rc;
    Op op; op.kind = OP_SE;
    float *d_w1 = nullptr, *d_b1 = nullptr, *d_w2 = nullptr, *d_b2 = nullptr;
    rc = net_upload(net, &d_w1, std::vector<float>(fc1_weight, fc1_weight + (size_t)squeeze * channels)); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b1, std::vector<float>(fc1_bias, fc1_bias + squeeze)); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_w2, std::vector<float>(fc2_weight, fc2_weight + (size_t)channels * squeeze)); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b2, std::vector<float>(fc2_bias, fc2_bias + channels)); if (rc != PIFPAF_OK) return rc;
    SeArgs& a = op.se;
    a.part = d_part; a.nslots = nc.nslots; a.C8 = C / 8; a.inv_hw = 1.0f / (float)(tin.h * tin.w);
    a.channels = channels; a.squeeze = squeeze;
    a.w1 = d_w1; a.b1 = d_b1; a.w2 = d_w2; a.b2 = d_b2;
    a.wproj = d_wproj; a.n_pad = gop.g.block_n * gop.g.n_blocks; a.k_total = gop.g.ldw;
    a.wimg = const_cast<__nv_bfloat16*>(gop.g.wgt);
    op.flops_per_image = 4.0 * channels * squeeze + (double)a.n_pad * a.k_total;
    op.bytes_per_image = (double)nc.nslots * C * 4.0 + (double)a.n_pad * a.k_total * 2.0;
    op.weight_bytes = (2.0 * channels * squeeze + channels + squeeze) * 4.0 + (double)a.n_pad * a.k_total * 4.0;
    net->ops.push_back(op);
    net->ops.push_back(gop);
    return PIFPAF_OK;
}

int pifpaf_net_dw_conv1x1_scatter(pifpaf_net_t* net, int32_t in_tensor, int32_t in_col_off, int32_t channels,
                                  int32_t kernel, int32_t stride, int32_t pad,
                                  const float* dw_weight, const float* dw_bias, int32_t dw_relu,
                                  int32_t n_out, const float* weight, const float* bias, int32_t relu,
                                  int32_t n_pieces, const int32_t* piece_col0, const int32_t* piece_count,
                                  const int32_t* piece_tensor, const int32_t* piece_tensor_col) {
    PIFPAF_CHECK_ARG(net != nullptr && dw_weight != nullptr && weight != nullptr && piece_col0 && piece_count &&
                     piece_tensor && piece_tensor_col, "null argument");
    const int nt = (int)net->tensors.size();
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < nt, "bad tensor id");
    PIFPAF_CHECK_ARG(kernel == 5 && stride == 1 && pad == 2, "the fused depthwise -> 1x1 op covers 5x5, stride 1, pad 2");
    PIFPAF_CHECK_ARG(n_out >= 16 && n_out % 16 == 0 && n_out <= 512 && n_pieces >= 1, "n_out: multiple of 16, at most 512");
    const Tensor& tin = net->tensors[in_tensor];
    const int C = pad8(channels);
    PIFPAF_CHECK_ARG(in_col_off % 8 == 0 && in_col_off + C <= tin.c, "depthwise column window");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    Op op; op.kind = OP_FUSED;
    // depthwise weights [C][25] -> tap-major [25][C]
    std::vector<float> dww((size_t)25 * C, 0.f), dwb(C, 0.f);
    for (int c = 0; c < channels; c++) {
        for (int t = 0; t < 25; t++) dww[(size_t)t * C + c] = dw_weight[(size_t)c * 25 + t];
        dwb[c] = dw_bias ? dw_bias[c] : 0.f;
    }
    float *d_dww = nullptr, *d_dwb = nullptr;
    int rc = net_upload(net, &d_dww, dww); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_dwb, dwb); if (rc != PIFPAF_OK) return rc;
    // 1x1 weights [n_out][channels] -> bf16 [n_pad][k_pad]
    FusedArgs& f = op.fu;
    f.n_halves = n_out > 256 ? 2 : 1;
    f.n_pad = f.n_halves == 2 ? (n_out + 31) / 32 * 32 : n_out;
    f.half_n = f.n_pad / f.n_halves;
    f.acc_stages = 2 * f.n_pad <= 512 ? 2 : 1;
    f.dw_weight = d_dww; f.dw_bias = d_dwb; f.C = C; f.dw_relu = dw_relu; f.pad = pad;
    const int k_pad = C;
    std::vector<__nv_bfloat16> w((size_t)f.n_pad * k_pad, __float2bfloat16(0.f));
    long long nnz = 0; int n_real = 0;
    for (int n = 0; n < n_out; n++) {
        bool row = bias != nullptr && bias[n] != 0.f;
        for (int k = 0; k < channels; k++) {
            const float v = weight[(size_t)n * channels + k];
            w[(size_t)n * k_pad + k] = __float2bfloat16(v);
            if (v != 0.f) { nnz++; row = true; }
        }
        n_real += row ? 1 : 0;
    }
    std::vector<float> b(f.n_pad, 0.f);
    for (int n = 0; n < n_out; n++) b[n] = bias ? bias[n] : 0.f;
    __nv_bfloat16* d_w = nullptr; float* d_b = nullptr;
    rc = net_upload(net, &d_w, w); if (rc != PIFPAF_OK) return rc;
    rc = net_upload(net, &d_b, b); if (rc != PIFPAF_OK) return rc;
    // scatter table
    std::vector<DestGroup> groups((size_t)f.n_pad / 16, DestGroup{nullptr, 0, 0});
    int expect = 0;
    for (int i = 0; i < n_pieces; i++) {
        PIFPAF_CHECK_ARG(piece_col0[i] == expect && piece_count[i] >= 16 && piece_count[i] % 16 == 0,
                         "pieces must tile [0, n_out) in order, in multiples of 16 columns");
        PIFPAF_CHECK_ARG(piece_tensor[i] >= 0 && piece_tensor[i] < nt, "bad piece tensor id");
        const Tensor& to = net->tensors[piece_tensor[i]];
        PIFPAF_CHECK_ARG(to.h == tin.h && to.w == tin.w, "stride 1 keeps the spatial shape");
        PIFPAF_CHECK_ARG(piece_tensor_col[i] >= 0 && piece_tensor_col[i] % 16 == 0 &&
                         piece_tensor_col[i] + piece_count[i] <= to.c, "piece window outside its tensor");
        for (int c = 0; c < piece_count[i]; c += 16)
            groups[(size_t)(expect + c) / 16] = DestGroup{to.data + piece_tensor_col[i] + c, to.c, 0};
        expect += piece_count[i];
    }
    PIFPAF_CHECK_ARG(expect == n_out, "pieces must cover all n_out columns");
    DestGroup* d_groups = nullptr;
    rc = net_upload(net, &d_groups, groups); if (rc != PIFPAF_OK) return rc;

    GemmArgs& g = op.g;
    g.N = n_out; g.K = C; g.block_n = f.n_pad; g.n_blocks = 1;
    g.num_k_blocks = (C + BK - 1) / BK;
    g.bias = d_b; g.mode = MODE_SCATTER; g.relu = relu; g.dest = d_groups;
    g.conv_k = kernel; g.conv_stride = stride; g.conv_pad = pad; g.conv_cblocks = g.num_k_blocks;
    g.Hi = tin.h; g.Wi = tin.w; g.Ho = tin.h; g.Wo = tin.w;
    g.tiles_x = (g.Wo + PW - 1) / PW; g.tiles_y = (g.Ho + PH - 1) / PH;
    op.a_tensor = in_tensor; op.rows_per_image = g.Ho * g.Wo; op.tiles_per_image = g.tiles_x * g.tiles_y;
    // ring depths: as deep as the shared memory allows, windows first (their TMA has the longest latency)
    // (an A stage is written only after the depthwise warps hold their results in registers, so one A stage costs
    // little; a single B stage would expose the weight TMA latency in every K block)
    // (an A stage is written only after the depthwise warps hold their results in registers, so one A stage costs
    // little; a single B stage would expose the weight TMA latency in every K block)
    const int cand[][3] = {{3, 3, 2}, {3, 2, 2}, {2, 2, 2}, {2, 1, 2}, {2, 2, 1}, {1, 1, 1}};
    bool fits = false;
    for (const auto& c : cand) {
        if (fused_smem_bytes(c[0], c[1], c[2], f.n_pad, C) <= GEMM_SMEM_BUDGET) {
            f.ws = c[0]; f.as = c[1]; f.bs = c[2]; fits = true; break;
        }
    }
    PIFPAF_CHECK_ARG(fits, "fused depthwise -> 1x1 op does not fit in shared memory");
    op.smem = fused_smem_bytes(f.ws, f.as, f.bs, f.n_pad, C);
    op.n_real = n_real;
    op.flops_per_image = 2.0 * (double)op.rows_per_image * ((double)nnz + 25.0 * channels);
    op.bytes_per_image = (double)op.rows_per_image * (channels + n_real) * 2.0;     // dw input once + 1x1 output once
    op.weight_bytes = (double)nnz * 2.0 + 25.0 * channels * 4.0;
    using T = DwTile<1, PH, PW, 4, 1>;
    rc = make_tmap_dw(&op.tmap_dw, tin.data + in_col_off, (uint64_t)C, (uint64_t)tin.w, (uint64_t)tin.h,
                      (uint64_t)net->max_batch, (uint64_t)tin.c, T::IW, T::IH);
    if (rc != PIFPAF_OK) return rc;
    rc = make_tmap(&op.tmap_b, d_w, (uint64_t)f.n_pad, (uint64_t)k_pad, (uint64_t)k_pad, (uint32_t)f.half_n);
    if (rc != PIFPAF_OK) return rc;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_heads(pifpaf_net_t* net, int32_t in_tensor, int32_t k_cols, int32_t n_heads,
                     const int32_t* n_fields, const int32_t* n_comp, const int32_t* comp_ops,
                     const float* weight, const float* bias) {
    return pifpaf_net_heads_upsampled(net, in_tensor, k_cols, n_heads, n_fields, n_comp, comp_ops, 1, weight, bias);
}

int pifpaf_net_heads_upsampled(pifpaf_net_t* net, int32_t in_tensor, int32_t k_cols, int32_t n_heads,
                               const int32_t* n_fields, const int32_t* n_comp, const int32_t* comp_ops,
                               int32_t upsample_stride, const float* weight, const float* bias) {
    PIFPAF_CHECK_ARG(net != nullptr && weight != nullptr && n_fields && n_comp && comp_ops, "null argument");
    PIFPAF_CHECK_ARG(n_heads >= 1 && n_heads <= 4, "1..4 heads supported");
    PIFPAF_CHECK_ARG(upsample_stride >= 1 && upsample_stride <= 8, "upsample_stride must be in [1, 8]");
    PIFPAF_CHECK_ARG(in_tensor >= 0 && in_tensor < (int)net->tensors.size(), "bad tensor id");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    const Tensor& tin = net->tensors[in_tensor];
    const int up = upsample_stride, up2 = up * up;
    // heads.py:336-343: low_cut = (up - 1) / 2, high_cut = ceil((up - 1) / 2)
    const int low = (up - 1) / 2, high = up / 2;
    const int out_h = tin.h * up - low - high, out_w = tin.w * up - low - high;
    PIFPAF_CHECK_ARG(out_h >= 1 && out_w >= 1, "feature map too small for this upsample_stride");
    int n_total = 0;
    for (int i = 0; i < n_heads; i++) n_total += n_fields[i] * n_comp[i] * up2;
    Op op; op.kind = OP_GEMM;
    int rc = emit_gemm(net, op, in_tensor, 0, k_cols, n_total, weight, bias);
    if (rc != PIFPAF_OK) return rc;
    GemmArgs& g = op.g;
    g.mode = MODE_HEADS; g.relu = 0;
    op.bytes_per_image += (double)out_h * out_w * (op.n_real / up2) * 4.0;
    std::vector<HeadCol> cols((size_t)g.block_n * g.n_blocks, HeadCol{0, 0, 0, 0});
    int col = 0, op_off = 0;
    for (int i = 0; i < n_heads; i++) {
        for (int f = 0; f < n_fields[i]; f++)
            for (int c = 0; c < n_comp[i]; c++)
                for (int dy = 0; dy < up; dy++)
                    for (int dx = 0; dx < up; dx++)
                        cols[col++] = HeadCol{i, f * n_comp[i] + c, comp_ops[op_off + c], (dy << 8) | dx};
        op_off += n_comp[i];
        net->head_fields[i] = n_fields[i]; net->head_comp[i] = n_comp[i];
        net->head_elems[i] = (size_t)net->max_batch * n_fields[i] * n_comp[i] * out_h * out_w;
        rc = net_alloc(net, &net->head_out[0][i], net->head_elems[i], true);
        if (rc != PIFPAF_OK) return rc;
        g.head_base[i] = net->head_out[0][i];
        g.head_planes[i] = n_fields[i] * n_comp[i];
    }
    HeadCol* d_cols = nullptr;
    rc = net_upload(net, &d_cols, cols); if (rc != PIFPAF_OK) return rc;
    g.head_cols = d_cols;
    g.hw = tin.h * tin.w; g.w = tin.w;
    g.up = up; g.up_low = low; g.out_h = out_h; g.out_w = out_w;
    net->n_heads = n_heads; net->head_h = out_h; net->head_w = out_w;
    rc = plan_gemm_pair(net, op); if (rc != PIFPAF_OK) return rc;
    net->ops.push_back(op);
    return PIFPAF_OK;
}

int pifpaf_net_head_output(pifpaf_net_t* net, int32_t head, float** dev_ptr,
                           int32_t* n_fields, int32_t* n_comp, int32_t* h, int32_t* w) {
    PIFPAF_CHECK_ARG(net != nullptr && head >= 0 && head < net->n_heads, "bad head index");
    if (dev_ptr) *dev_ptr = net->head_out[net->head_cur][head];     // the set the last forward wrote
    if (n_fields) *n_fields = net->head_fields[head];
    if (n_comp) *n_comp = net->head_comp[head];
    if (h) *h = net->head_h;
    if (w) *w = net->head_w;
    return PIFPAF_OK;
}

struct RawImages { const uint8_t* images; float mean[3], stdev[3]; };

static int net_forward_impl(pifpaf_net_t* net, const float* images_dev, int32_t batch, int32_t gemm_impl,
                            cudaStream_t st, cudaEvent_t* events, const RawImages* u8 = nullptr) {
    PIFPAF_CHECK_ARG(net != nullptr, "null argument");
    PIFPAF_CHECK_ARG(images_dev != nullptr || u8 != nullptr || net->in_h == 0, "images pointer is null");
    PIFPAF_CHECK_ARG(batch >= 1 && batch <= net->max_batch, "batch exceeds max_batch");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    if (!net->setup_synced) {
        // tensors were zero-filled and weights uploaded on the legacy default stream at emit time; `st` may be a
        // non-blocking stream that does not order itself behind it
        PIFPAF_CUDA_TRY(cudaDeviceSynchronize());
        net->setup_synced = true;
    }
    if (net->head_buffers == 2) net->head_cur ^= 1;
    const int n_sm = net->sm_limit > 0 ? std::min(net->sm_limit, net->n_sm) : net->n_sm;
    int op_index = 0;
    // PDL between consecutive ops (not in the per-op timing pass: the events would sit between the launches; not for
    // the first op: its predecessor in the stream is a copy or another forward's decode, not one of these kernels)
    const bool pdl_on = net->pdl && events == nullptr && gemm_impl == 0;
    for (Op& op : net->ops) {
        if (events) PIFPAF_CUDA_TRY(cudaEventRecord(events[op_index], st));
        const bool pdl = pdl_on && op_index > 0;
        op_index++;
        if (op.kind == OP_INPUT_CONV) {
            InConvArgs a = op.ic;
            a.in = images_dev; a.B = batch;
            const long long total = (long long)batch * a.Hout * a.Wout;
            const int grid = (int)std::min<long long>((total + 255) / 256, (long long)n_sm * 16);
            const size_t smem = sizeof(float) * ((size_t)3 * a.kernel * a.kernel * a.C8 * 8 + a.C8 * 8 + 3 * 256);
            if (u8 != nullptr) {
                a.in_u8 = u8->images;
                for (int c = 0; c < 3; c++) { a.mean[c] = u8->mean[c]; a.stdev[c] = u8->stdev[c]; }
                if (a.relu >= 2) k_input_conv<3, true, true><<<grid, 256, smem, st>>>(a);
                else if (a.kernel == 3) k_input_conv<3, true><<<grid, 256, smem, st>>>(a);
                else if (a.kernel == 7) k_input_conv<7, true><<<grid, 256, smem, st>>>(a);
                else if (a.kernel == 5) k_input_conv<5, true><<<grid, 256, smem, st>>>(a);
                else k_input_conv<1, true><<<grid, 256, smem, st>>>(a);
            } else if (a.relu >= 2) k_input_conv<3, false, true><<<grid, 256, smem, st>>>(a);
            else if (a.kernel == 3) k_input_conv<3, false><<<grid, 256, smem, st>>>(a);
            else if (a.kernel == 7) k_input_conv<7, false><<<grid, 256, smem, st>>>(a);
            else if (a.kernel == 5) k_input_conv<5, false><<<grid, 256, smem, st>>>(a);
            else k_input_conv<1, false><<<grid, 256, smem, st>>>(a);
            PIFPAF_LAUNCH_CHECK();
        } else if (op.kind == OP_FUSED) {
            PIFPAF_CHECK_ARG(gemm_impl == 0, "the fused depthwise -> 1x1 op has no SIMT debug variant (compile the net with fuse_dw=False)");
            GemmArgs g = op.g;
            g.M = batch * op.rows_per_image;
            g.m_blocks = batch * op.tiles_per_image;
            const int grid = std::min(g.m_blocks, n_sm);
            PIFPAF_CUDA_TRY(launch_k(pdl, k_dw_gemm<1>, dim3(grid), dim3(FD_THREADS), op.smem, st, op.tmap_dw, op.tmap_b, g, op.fu));
            PIFPAF_LAUNCH_CHECK();
        } else if (op.kind == OP_SE) {
            const size_t smem = sizeof(float) * (2 * (size_t)op.se.C8 * 8 + op.se.squeeze);
            k_se<<<batch, SE_THREADS, smem, st>>>(op.se);
            PIFPAF_LAUNCH_CHECK();
        } else if (op.kind == OP_DW) {
            DwArgs a = op.dw;
            a.B = batch;
            if (op.dw_nc) {
                DwNcArgs x = op.dwnc; int block = 0;
                plan_dw_nc(a, &x, &block);
                x.se_part = op.dwnc.se_part;
                const dim3 grid((unsigned)x.nslots, (unsigned)batch);
                if (a.kernel == 3 && a.stride == 1) k_dwconv_nc<3, 1><<<grid, block, 0, st>>>(a, x);
                else if (a.kernel == 3) k_dwconv_nc<3, 2><<<grid, block, 0, st>>>(a, x);
                else if (a.stride == 1) k_dwconv_nc<5, 1><<<grid, block, 0, st>>>(a, x);
                else k_dwconv_nc<5, 2><<<grid, block, 0, st>>>(a, x);
            } else if (op.dw_tc && gemm_impl == 0) {
                const int cblks = (a.C8 + 7) / 8;
                const long long total = (long long)batch * ((a.Hout + DT_TH - 1) / DT_TH) * ((a.Wout + DT_TW - 1) / DT_TW) * cblks;
                const int grid = (int)std::min<long long>(total, (long long)n_sm);
                DwTcArgs x; x.pwid = a.stride == 1 ? net->dw_tc_pwid : DwTc<2>::PWID; x.base_off_mode = net->dw_tc_bo;
                if (a.stride == 1) {
                    const size_t plane = (size_t)((DwTc<1>::IH * x.pwid * 128 + 1023) / 1024) * 1024;
                    const size_t smem = DwTc<1>::STAGES * plane + DT_B_BYTES + 64 * 4 + 128 + 1024;
                    PIFPAF_CUDA_TRY(launch_k(pdl, k_dwconv5_tc<1>, dim3(grid), dim3(DT_THREADS), smem, st, op.tmap_dw_tc, a, x));
                } else {
                    PIFPAF_CUDA_TRY(launch_k(pdl, k_dwconv5_tc<2>, dim3(grid), dim3(DT_THREADS), (size_t)DwTc<2>::SMEM, st,
                                             op.tmap_dw_tc, a, x));
                }
            } else if (op.dw_tma && gemm_impl == 0) {
                const int cblks = (a.C8 + 7) / 8;
                // persistent grid == resident CTAs (stride 1: 2 per SM, stride 2: 1 per SM by shared memory)
                if (a.stride == 1) {
                    const long long total = (long long)batch * ((a.Hout + DW1_TH - 1) / DW1_TH) *
                                            ((a.Wout + DW1_TW - 1) / DW1_TW) * cblks;
                    const int grid = (int)std::min<long long>(total, (long long)n_sm * 2);
                    PIFPAF_CUDA_TRY(launch_k(pdl, k_dwconv5_tma<1, DW1_TH, DW1_TW, 4, 3, false>, dim3(grid), dim3(DwS1::THREADS),
                                             (size_t)DwS1::SMEM, st, op.tmap_dw, a));
                } else {
                    const long long total = (long long)batch * ((a.Hout + DW2_TH - 1) / DW2_TH) *
                                            ((a.Wout + DW2_TW - 1) / DW2_TW) * cblks;
                    const int grid = (int)std::min<long long>(total, (long long)n_sm);
                    // channel-block-fastest order with the weights staged in shared memory while they fit
                    const size_t smem_cf = (size_t)DwS2::SMEM + (size_t)26 * a.C8 * 8 * sizeof(float);
                    if (net->dw_cbf && cblks > 1 && smem_cf <= 226 * 1024)
                        PIFPAF_CUDA_TRY(launch_k(pdl, k_dwconv5_tma<2, DW2_TH, DW2_TW, 4, 2, true>, dim3(grid), dim3(DwS2::THREADS),
                                                 smem_cf, st, op.tmap_dw, a));
                    else
                        PIFPAF_CUDA_TRY(launch_k(pdl, k_dwconv5_tma<2, DW2_TH, DW2_TW, 4, 2, false>, dim3(grid), dim3(DwS2::THREADS),
                                                 (size_t)DwS2::SMEM, st, op.tmap_dw, a));
                }
            } else if (a.kernel == 5 && (a.stride == 1 || a.stride == 2)) {
                const long long total = (long long)batch * ((a.Hout + DW_OY - 1) / DW_OY) * DW_OY *
                                        ((a.Wout + DW_OX - 1) / DW_OX) * a.C8;
                const int grid = (int)std::min<long long>((total + 255) / 256, (long long)n_sm * 64);
                if (a.stride == 1) k_dwconv5<1><<<grid, 256, 0, st>>>(a);
                else k_dwconv5<2><<<grid, 256, 0, st>>>(a);
            } else {
                const long long total = (long long)batch * a.Hout * a.Wout * a.C8;
                const int grid = (int)std::min<long long>((total + 255) / 256, (long long)n_sm * 32);
                k_dwconv<<<grid, 256, 0, st>>>(a);
            }
            PIFPAF_LAUNCH_CHECK();
        } else {
            GemmArgs g = op.g;
            g.debug = net->gemm_debug;
            if (g.mode == MODE_HEADS)
                for (int i = 0; i < net->n_heads; i++) g.head_base[i] = net->head_out[net->head_cur][i];
            g.M = batch * op.rows_per_image;
            g.m_blocks = g.conv_k > 0 ? batch * op.tiles_per_image : (g.M + BM - 1) / BM;
            const bool ext = g.relu >= 2 || g.w_img_rows > 0;
            if (gemm_impl == 1) {
                const long long jobs = (long long)g.m_blocks * 4 * (g.n_blocks * g.block_n / CHUNK);
                const int grid = (int)std::min<long long>((jobs + 3) / 4, (long long)n_sm * 16);
                k_gemm_simt<<<grid, 128, 0, st>>>(g);
            } else if (op.pair) {
                g.pair = 1; g.pair_stages = op.pair_stages; g.b_resident = op.pair_resident;
                const int m2 = (g.M + 2 * BM - 1) / (2 * BM);
                const int max_pairs = std::max(1, n_sm / 2);
                int pairs = std::min(max_pairs, m2 * g.n_blocks);
                if (g.b_resident) pairs = std::max(1, std::min(max_pairs / g.n_blocks, m2)) * g.n_blocks;
                PIFPAF_CUDA_TRY(launch_kc(pdl, 2, ext ? k_gemm_tc2<true> : k_gemm_tc2<false>, dim3(2 * pairs), dim3(GEMM_THREADS), op.pair_smem, st, op.tmap_a,
                                          op.tmap_bh, g));
            } else {
                const int tiles = g.m_blocks * g.n_blocks;
                int grid = std::min(tiles, n_sm);
                if (g.b_resident) grid = std::max(1, std::min(n_sm / g.n_blocks, g.m_blocks)) * g.n_blocks;
                // multicast pairs need at least one whole cluster and whole clusters only (grid is a multiple of n_blocks == 2)
                PIFPAF_CUDA_TRY(launch_kc(pdl, g.mc ? 2 : 1, ext ? k_gemm_tc<true> : k_gemm_tc<false>, dim3(grid), dim3(GEMM_THREADS), op.smem, st, op.tmap_a,
                                          op.tmap_b, (g.src_tma || g.mc) ? op.tmap_src : op.tmap_a, g));
            }
            PIFPAF_LAUNCH_CHECK();
        }
    }
    if (events) PIFPAF_CUDA_TRY(cudaEventRecord(events[op_index], st));
    return PIFPAF_OK;
}

int pifpaf_net_forward(pifpaf_net_t* net, const float* images_dev, int32_t batch, int32_t gemm_impl,
                       void* stream_v) {
    return net_forward_impl(net, images_dev, batch, gemm_impl, reinterpret_cast<cudaStream_t>(stream_v), nullptr);
}

int pifpaf_net_forward_u8(pifpaf_net_t* net, const uint8_t* images_nhwc_dev, int32_t batch, const float* mean,
                          const float* stdev, int32_t gemm_impl, void* stream_v) {
    PIFPAF_CHECK_ARG(images_nhwc_dev != nullptr && mean != nullptr && stdev != nullptr, "null argument");
    RawImages raw;
    raw.images = images_nhwc_dev;
    for (int c = 0; c < 3; c++) {
        PIFPAF_CHECK_ARG(stdev[c] > 0.f, "std must be positive");
        raw.mean[c] = mean[c]; raw.stdev[c] = stdev[c];
    }
    return net_forward_impl(net, nullptr, batch, gemm_impl, reinterpret_cast<cudaStream_t>(stream_v), nullptr, &raw);
}

int pifpaf_net_forward_timed(pifpaf_net_t* net, const float* images_dev, int32_t batch, int32_t gemm_impl,
                             void* stream_v, float* op_ms, int32_t* op_kind, double* op_flops, double* op_bytes) {
    PIFPAF_CHECK_ARG(net != nullptr && op_ms != nullptr, "null argument");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream_v);
    const size_t n = net->ops.size();
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) PIFPAF_CUDA_TRY(cudaEventCreate(&e));
    int rc = net_forward_impl(net, images_dev, batch, gemm_impl, st, ev.data());
    if (rc == PIFPAF_OK) {
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { pifpaf::set_error("forward failed: %s", cudaGetErrorString(e)); rc = PIFPAF_E_CUDA; }
    }
    for (size_t i = 0; i < n && rc == PIFPAF_OK; i++) {
        cudaEventElapsedTime(&op_ms[i], ev[i], ev[i + 1]);
        const Op& op = net->ops[i];
        if (op_kind) op_kind[i] = op.kind == OP_INPUT_CONV ? 0 : op.kind == OP_GEMM ? 1 : op.kind == OP_DW ? 2 : op.kind == OP_FUSED ? 3 : 4;
        if (op_flops) op_flops[i] = op.flops_per_image * batch;
        if (op_bytes) op_bytes[i] = op.bytes_per_image * batch + op.weight_bytes;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return rc;
}

int pifpaf_net_tap_tensor(pifpaf_net_t* net, int32_t id, int32_t batch, float* out, int64_t out_elems) {
    PIFPAF_CHECK_ARG(net != nullptr && id >= 0 && id < (int)net->tensors.size(), "bad tensor id");
    const Tensor& t = net->tensors[id];
    const long long n = (long long)batch * t.h * t.w * t.c;
    PIFPAF_CHECK_ARG(out != nullptr && out_elems >= n && batch <= net->max_batch, "output buffer too small");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    float* d_tmp = nullptr;
    PIFPAF_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_tmp), sizeof(float) * n));
    k_bf16_to_f32<<<1024, 256>>>(t.data, d_tmp, n);
    pifpaf::count_launch();
    cudaError_t e = cudaMemcpy(out, d_tmp, sizeof(float) * n, cudaMemcpyDeviceToHost);
    cudaFree(d_tmp);
    if (e != cudaSuccess) { pifpaf::set_error("tap copy failed: %s", cudaGetErrorString(e)); return PIFPAF_E_CUDA; }
    return PIFPAF_OK;
}

int pifpaf_net_set_tensor(pifpaf_net_t* net, int32_t id, int32_t batch, const float* data, int64_t n_elems) {
    PIFPAF_CHECK_ARG(net != nullptr && id >= 0 && id < (int)net->tensors.size(), "bad tensor id");
    const Tensor& t = net->tensors[id];
    const long long n = (long long)batch * t.h * t.w * t.c;
    PIFPAF_CHECK_ARG(data != nullptr && n_elems == n && batch <= net->max_batch, "input size mismatch");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    float* d_tmp = nullptr;
    PIFPAF_CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&d_tmp), sizeof(float) * n));
    cudaError_t e = cudaMemcpy(d_tmp, data, sizeof(float) * n, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        k_f32_to_bf16<<<1024, 256>>>(d_tmp, t.data, n);
        pifpaf::count_launch();
        e = cudaDeviceSynchronize();
    }
    cudaFree(d_tmp);
    if (e != cudaSuccess) { pifpaf::set_error("set_tensor failed: %s", cudaGetErrorString(e)); return PIFPAF_E_CUDA; }
    return PIFPAF_OK;
}

int pifpaf_net_set_head_buffers(pifpaf_net_t* net, int32_t n_buffers) {
    PIFPAF_CHECK_ARG(net != nullptr && (n_buffers == 1 || n_buffers == 2), "n_buffers must be 1 or 2");
    PIFPAF_CUDA_TRY(cudaSetDevice(net->device));
    if (n_buffers == 2) {
        for (int i = 0; i < net->n_heads; i++) {
            if (net->head_out[1][i] != nullptr) continue;
            int rc = net_alloc(net, &net->head_out[1][i], net->head_elems[i], true);
            if (rc != PIFPAF_OK) return rc;
        }
        net->setup_synced = false;
    } else {
        net->head_cur = 0;
    }
    net->head_buffers = n_buffers;
    return PIFPAF_OK;
}

int pifpaf_net_set_sm_limit(pifpaf_net_t* net, int32_t n_sm) {
    PIFPAF_CHECK_ARG(net != nullptr && n_sm >= 0, "bad argument");
    net->sm_limit = n_sm;
    return PIFPAF_OK;
}

double pifpaf_net_flops_per_image(pifpaf_net_t* net) {
    if (!net) return 0.0;
    double f = 0.0;
    for (const Op& op : net->ops) f += op.flops_per_image;
    return f;
}

int32_t pifpaf_net_num_ops(pifpaf_net_t* net) { return net ? (int32_t)net->ops.size() : 0; }

}  // extern "C"
