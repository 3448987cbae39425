// Head 1x1 convolution fused with the YOLO decode + confidence filter + stream compaction (sm_100a, tcgen05).
//
// SURVEY.md section 8f-3: the producer of every head tensor is a dense contraction
//     head[b, o, y, x] = act( sum_c W[o, c] * X[b, c, y, x] + bias[o] )
// (reference models/yolov3_spp.py:86,99,111 -- ConvBlock = 1x1 conv + BatchNorm + LeakyReLU(0.1),
// models/yolo_base.py:19-44; models/yolov3_tiny.py:38,42 -- a plain nn.Conv2d with bias), C_in = 256..1024,
// 255 output channels.  Computing it here and decoding straight out of the accumulator removes the
// 340 B/anchor head tensor from HBM altogether: the only traffic left is one read of X.
//
// One persistent CTA per SM, warp-specialised:
//   warp 0      TMA producer   X tile  [32 channels] x [128 positions]  (one 3-D box = 4 atoms of 32 x 32,
//                                                                        SWIZZLE_128B_ATOM_32B)              = A, MN-major
//                              W tile  [NPAD rows]   x [32 channels]    (one 2-D box, SWIZZLE_128B)         = B, K-major
//   warp 1      MMA issuer     tcgen05.mma.cta_group::1.kind::tf32, M = 128 positions, N = NPAD (256) output channels,
//                              K = 8 per instruction; fp32 accumulators in TMEM, two accumulator stages (2 x 256 columns)
//   warps 2..13 epilogue       one warp per (TMEM lane quarter, anchor): tcgen05.ld 32x32b, a thread owns one position (TMEM
//                              lane) and walks its anchor's 85 output channels (TMEM columns): bias + LeakyReLU, then
//                              exactly the per-anchor arithmetic of decode_compact_kernel (decode.cu): running (max, 2nd
//                              max, first arg-max) over the class logits, score, thresholds, box decode, warp-aggregated
//                              candidate emission.
// All scales of a model run in one launch (tiles dealt round-robin, heaviest scale first).  A CTA-pair variant
// (cta_group::2) follows the single-CTA kernel.
// The TF32 tensor-core product rounds the operands to 10 mantissa bits (what cuDNN does for the reference's fp32
// convolution on this GPU with torch's default allow_tf32), so the head values differ from an fp32 CPU convolution by
// ~1e-3 relative; everything after the accumulator is bit-identical to decode_compact_kernel fed with the head tensor
// this kernel can also write out (head_out) -- that is the parity test.
//
// fp16 / bf16 feature maps (YOLO_B200_HEAD_F16 / _BF16, template parameter DT): the same kernel with a 16-bit main loop.
// Only the producer, the MMA issuer and the loader warps differ; the epilogue reads the same fp32 accumulators.
//   X tile  [64 channels] x [128 positions]: two 64-position atoms of 64 x 128-byte rows (8 KB each), plain SWIZZLE_128B
//           (one 3-D box of 64 x 64 x 2, or a 2-D box of 64 x 64 per atom)                    = A, MN-major
//   W tile  [NPAD rows] x [64 channels]: one 128-byte row per output channel, SWIZZLE_128B     = B, K-major
//   tcgen05.mma.cta_group::1.kind::f16 (A and B of the feature map's type, fp32 accumulators), K = 16 per instruction.
// A stage is 16 KB of X + NPAD x 128 bytes of W: the same 48 KB as the fp32 stage.  Planes without a 16-byte pitch
// (plane % 8 != 0) but with 4-byte aligned rows (even planes) are filled by the loader warps with 8-byte (plane % 4 == 0)
// or 4-byte copies; odd planes are padded by the host first (yolo_b200_pad_planes_16).
//
// channels_last feature maps (YOLO_B200_HEAD_NHWC, HeadParams.nhwc, uniform per launch): X is a row-major
// (B*plane, c_in) matrix, so A is K-major like W.  One 3-D box of (c_in, plane, batch) per k-block -- BK channels (128
// bytes) x 128 positions x 1 image, SWIZZLE_128B, positions past the plane zero-filled -- and the A descriptor of B
// (SBO 1 KB, +32 bytes per MMA K step) with the instruction descriptor's A-major bit clear.  Every plane size is read in
// place (no loader warps, no padded copy); the W ring, the epilogue and head_out are unchanged.
#include <cuda.h>          // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)

#include "common.cuh"

namespace yb {
namespace hd {

constexpr int kBK = 32;                    // channels per pipeline stage = one 128-byte swizzle span of a W row
constexpr int kM = 128;                    // positions per tile = UMMA M = TMEM lanes
#ifndef YB_HEAD_STAGES
#define YB_HEAD_STAGES 4
#endif
constexpr int kStages = YB_HEAD_STAGES;
constexpr int kProducerThreads = 64;      // warp 0: TMA, warp 1: MMA; then 4 epilogue warps per anchor
constexpr int kAtomBytes = 32 * kBK * 4;   // one [32 channels][32 positions] atom of X: 4 KB
constexpr int kABytes = 4 * kAtomBytes;    // 16 KB
constexpr int kMaxN = 256;
constexpr int kTmemCols = 512;
constexpr int kWatchdog = 0x100;           // added to *overflow when a pipeline wait times out (never in a correct run)
// 16-bit main loop: a k-block is 64 channels (one 128-byte W row), an X atom 64 positions x 64 channel rows
constexpr int kBK16 = 64;
constexpr int kAtomBytes16 = 64 * kBK16 * 2;     // 8 KB; two atoms = kABytes
enum : int { kDtF32 = 0, kDtF16 = 1, kDtBF16 = 2 };

struct HeadScale {                         // one detection scale = one head convolution
    alignas(64) CUtensorMap tmap_x;        // [batch*c_in rows][plane] fp32 (row pitch >= plane), box 32 positions x 32 rows
    alignas(64) CUtensorMap tmap_x3;       // 3-D view of X: [32 positions][batch*c_in rows][plane/32 atoms], box 32 x 32 x 4
    alignas(64) CUtensorMap tmap_w;        // [NPAD rows][c_in] fp32, box 32 channels x NPAD rows
    alignas(64) CUtensorMap tmap_w2;       // the same tensor, box 32 channels x NPAD/2 rows (CTA-pair kernel)
    float bias[kMaxN];
    float slope;                           // LeakyReLU negative slope; 1 = no activation
    int c_in, kblocks;
    int ny, nx, plane, row_off;
    int tiles_per_img;                     // 128-position tiles per image
    int first_tile;                        // first global tile index of this scale (scales are ordered heaviest first)
    int use_x3;                            // tmap_x3 is valid
    int manual;                            // planes without a 16-byte pitch (19x19, 13x13): no tensor map for X, loader warps
    const float* x;                        // ... fill the stages from here with 4-byte asynchronous copies (16-bit elements
                                           // with YOLO_B200_HEAD_F16 / _BF16: 8- or 4-byte copies)
    float stride;
    float av[YOLO_B200_MAX_ANCHORS][2];
    float* head_out;                       // optional (batch, NA*(5+NC), ny, nx)
};

struct HeadParams {
    HeadScale sc[YOLO_B200_MAX_SCALES];
    int n_scales, batch, n_tiles;          // n_tiles: over all scales
    int nc;                                // classes (read by the kernels instantiated for a run-time class count)
    int pair_scale;                        // CTA-pair kernel: the one scale this launch works on
    float conf, min_wh;
    yolo_b200_box* cand_box;
    yolo_b200_meta* cand_meta;
    int cap;
    int32_t* count;
    int32_t* overflow;
    int emit;                              // 0: only write head_out (convolution only)
    int nhwc;                              // channels_last X (YOLO_B200_HEAD_NHWC): tmap_x is the 3-D (c_in, plane, batch)
                                           // map, one box per k-block, and A is K-major (read by the producer and the MMA thread)
    int skip_epilogue;                     // profiling bits (8 = the MMA thread only recycles the stages): 1 = epilogue warps only release the accumulator, 2 = W fetched
                                           // only for the first ring round, 4 = X fetched only for the first ring round
};

// ---- PTX helpers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
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
        : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must end the kernel with an error, never hang the GPU.  The bound is WALL-CLOCK time
// (%globaltimer, looked at every 64 K polls): 10 s without progress cannot be time-slicing, MPS or a debugger.  On
// expiry the kernel traps -- the launch fails and the next synchronisation on the stream reports it (the context is
// gone, so there is no softer way to tell the host; the role that gave up is left in *overflow for a post-mortem).
// BACKOFF: the epilogue warps wait for a whole main loop; sleeping between polls leaves their issue slots to the TMA and
// MMA issuing threads they share a scheduler with (ncu: 12-15 % of the kernel's instructions were barrier polling).
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
template <bool BACKOFF = false>
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int32_t* overflow, int who) {
    unsigned long long t0 = 0;
    for (uint32_t spins = 0; !mbar_try_wait(bar, parity); ++spins) {
        if constexpr (BACKOFF) __nanosleep(128);
        if ((spins & 0xffffu) == 0xffffu) {
            const unsigned long long now = global_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > 10000000000ull) {
                atomicMax(overflow, kWatchdog + who);
                __trap();
            }
        }
    }
}
__device__ __forceinline__ void tma_tile_g2s(uint32_t dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}
// 3-D tiled load: box = [32 positions] x [kBK channel rows] x [4 atoms] of the (position-in-atom, row, atom) view of X
__device__ __forceinline__ void tma_tile3_g2s(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
// 4-byte asynchronous copy global -> shared (LDGSTS) and its completion hook: the mbarrier receives one arrival (counted
// in its expected arrivals: .noinc) once every copy this thread issued so far has landed
__device__ __forceinline__ void cp_async4(uint32_t dst, const float* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// tcgen05.commit: the mbarrier receives one arrival once every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], tf32 inputs, fp32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], fp16 or bf16 inputs (the instruction descriptor says which), fp32 accumulate
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}

// Shared-memory matrix descriptor (tcgen05): start address, leading / stride byte offsets (16-byte units),
// descriptor version 1 (Blackwell), swizzle mode: 2 = SWIZZLE_128B (16-byte chunks, 8-row period),
// 1 = SWIZZLE_128B_BASE32B (32-byte chunks, 4-row period) -- the only layout the tensor core accepts for an MN-major
// 32-bit operand (measured: MN-major tf32 with the 16-byte-base swizzle yields all-zero accumulators,
// profiles/umma_probe.cu).
constexpr uint32_t kSw128 = 2, kSw128Base32 = 1;
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3fffu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32;
    d |= (uint64_t)1 << 46;            // version
    d |= (uint64_t)layout << 61;
    return d;
}
// the descriptor `fixed` (built with address 0) pointed at addr
__device__ __forceinline__ uint64_t smem_desc_at(uint64_t fixed, uint32_t addr) { return fixed | (uint64_t)((addr >> 4) & 0x3fffu); }
// Instruction descriptor: fp32 accumulator, tf32 A and B, A MN-major (positions contiguous), B K-major, M x N tile.
__host__ __device__ constexpr uint32_t instr_desc_tf32(int m, int n) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (0u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
// The same for kind::f16: A and B format 0 = F16, 1 = BF16 (fp32 accumulator, A MN-major, B K-major).
__host__ __device__ constexpr uint32_t instr_desc_f16(int m, int n, bool bf16) {
    return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | (1u << 15) | (0u << 16) | ((uint32_t)(n >> 3) << 17) |
           ((uint32_t)(m >> 4) << 24);
}

// TMEM -> registers: N consecutive columns of this thread's lane (the column may be any offset inside the allocation).
// The loads are asynchronous; tmem_wait_ld makes all of them visible.  ptxas tracks the destination registers of LDTM
// on the scoreboard; the empty asm statements after the wait keep the compiler from moving a use above it.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld2(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld1(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[0]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void pin_after_wait(uint32_t* r) {
#pragma unroll
    for (int i = 0; i < N; ++i) asm volatile("" : "+r"(r[i]));
}
// all N columns starting at taddr, as the fewest power-of-two loads (16-column pieces first)
template <int N>
__device__ __forceinline__ void tmem_ld_all(uint32_t taddr, uint32_t* r) {
    constexpr int F = N / 16;
#pragma unroll
    for (int c = 0; c < F; ++c) tmem_ld16(taddr + 16u * c, r + 16 * c);
    int off = 16 * F;
    if constexpr ((N & 8) != 0) { tmem_ld8(taddr + off, r + off); off += 8; }
    if constexpr ((N & 4) != 0) { tmem_ld4(taddr + off, r + off); off += 4; }
    if constexpr ((N & 2) != 0) { tmem_ld2(taddr + off, r + off); off += 2; }
    if constexpr ((N & 1) != 0) { tmem_ld1(taddr + off, r + off); }
}

// bias + LeakyReLU (nn.LeakyReLU: x if x > 0 else slope * x; for 0 <= slope <= 1 that is max(x, slope * x)).
// LEAKY = false is the slope == 1 case (a plain convolution head): max(v, v * 1) == v, two instructions less per element.
template <bool LEAKY>
__device__ __forceinline__ float activate(float acc, float bias, float slope) {
    const float v = __fadd_rn(acc, bias);
    if constexpr (LEAKY) return fmaxf(v, __fmul_rn(v, slope));
    else return v;
}

// Per-anchor epilogue; the same arithmetic, in the same order, as finish_anchor in decode.cu.  All 32 lanes call
// (tcgen05.ld and the ballots are warp collectives).  cls_taddr = TMEM address of this anchor's class-0 column of this
// thread's lane, cls_bias = its bias in shared memory.
template <bool LEAKY>
__device__ __forceinline__ void finish_anchor_tmem(const HeadParams& P, const HeadScale& S, int nc, bool active, int img, int a, int pos, int gx, int gy,
                                                   float t0, float t1, float t2, float t3, float t4,
                                                   float m, float m2, int idx, uint32_t cls_taddr, const float* cls_bias) {
    const float kSlack = 1.00003f;
    float so = 0.f, sm = 1.0f;
    bool pass = false, need = false;
    if (active) {
        so = sigmoidf_rn(t4);
        sm = (nc > 1) ? sigmoidf_rn(m) : 1.0f;                  // n_classes == 1: column 5 := 1 (yolo_layer.py:95-96)
        pass = so * sm * kSlack > P.conf;
        need = pass && nc > 1 && (sigmoidf_rn(m2) * kSlack >= sm);
    }
    float cls_conf = sm;
    int cls = idx;
    if (__any_sync(kFull, need)) {                 // exact class pick in sigmoid space (rescan_classes in decode.cu)
        float best = -1.0f;
        int bi = 0;
#pragma unroll 1
        for (int k = 0; k < nc; ++k) {
            uint32_t r;
            tmem_ld1(cls_taddr + k, &r);
            tmem_wait_ld();
            pin_after_wait<1>(&r);
            const float s = sigmoidf_rn(activate<LEAKY>(__uint_as_float(r), cls_bias[k], S.slope));
            if (s > best) { best = s; bi = k; }
        }
        if (need) { cls_conf = best; cls = bi; }
    }
    bool emit = false;
    yolo_b200_box box = {0.f, 0.f, 0.f, 0.f};
    float score = 0.f;
    if (pass) {
        score = __fmul_rn(so, cls_conf);                                  // utils.py:213
        if (score > P.conf) {                                             // utils.py:216
            const float w = decode_wh(t2, S.av[a][0], S.stride);
            const float h = decode_wh(t3, S.av[a][1], S.stride);
            if (w > P.min_wh && h > P.min_wh && finitef(w) && finitef(h)) {   // utils.py:217-218
                const float x = decode_xy(t0, (float)gx, S.stride);
                const float y = decode_xy(t1, (float)gy, S.stride);
                if (finitef(x) && finitef(y)) {
                    emit = true;
                    box = to_corners(x, y, w, h);                         // utils.py:231
                }
            }
        }
    }
    const int slot = warp_claim_slot(emit, img, P.count);
    if (emit) {
        if (slot < P.cap) {
            const int row = S.row_off + a * S.plane + pos;
            store_candidate(P.cand_box, P.cand_meta, (size_t)img * P.cap + slot, box, score, cls_conf, cls, row);
        } else {
            atomicMax(P.overflow, 1);
        }
    }
}

// Epilogue of one anchor for one TMEM lane (= position).  The anchor's 5+NC accumulator columns start at taddr_a (any
// column offset); all of them are requested at once -- one TMEM round trip per tile -- and then consumed from registers.
// The anchor index only enters through taddr_a / bias_a / hout_a, so the NA warps of a lane quarter run the same code
// (the first version had one unrolled copy per anchor and stalled on instruction fetch: profiles/r01_k_*).
// WRITE_HEAD / LEAKY are compile-time: the epilogue competes with the TMA and MMA issuing threads for issue slots (ncu:
// issue active 52 %, 1.1 warps "not selected" per issue), and the head_out stores and the LeakyReLU cost 3 + 2 of ~11
// instructions per element.
template <int NC, bool WRITE_HEAD, bool LEAKY>
__device__ __forceinline__ void epilogue_anchor(const HeadParams& P, const HeadScale& S, uint32_t taddr_a, const float* bias_a,
                                                float* hout_a, bool active, int img, int a, int pos) {
    constexpr int NO = NC + 5;
    uint32_t r[NO];
    tmem_ld_all<NO>(taddr_a, r);
    tmem_wait_ld();
    pin_after_wait<NO>(r);
    float t[5];
    float m = __int_as_float(0xff800000), m2 = m;
    int idx = 0;
#pragma unroll
    for (int ch = 0; ch < NO; ++ch) {
        const float v = activate<LEAKY>(__uint_as_float(r[ch]), bias_a[ch], S.slope);
        if constexpr (WRITE_HEAD) {
            if (hout_a && active) hout_a[(size_t)ch * S.plane] = v;
        }
        if (ch < 5) {
            t[ch] = v;
        } else if (NC > 1) {
            const bool up = v > m;
            m2 = up ? m : fmaxf(m2, v);
            idx = up ? (ch - 5) : idx;
            m = fmax_nan(m, v);
        }
    }
    if (P.emit) {
        const int gy = pos / S.nx, gx = pos - gy * S.nx;
        finish_anchor_tmem<LEAKY>(P, S, NC, active, img, a, pos, gx, gy, t[0], t[1], t[2], t[3], t[4], m, m2, idx, taddr_a + 5u, bias_a + 5);
    }
}

// The same epilogue for a class count known only at run time (any nc with NA * (5 + nc) <= 256): the five box / objectness
// columns first, then the class columns in 16-column pieces and a one-column tail -- never a column beyond the anchor's own.
template <bool WRITE_HEAD, bool LEAKY>
__device__ __forceinline__ void epilogue_anchor_generic(const HeadParams& P, const HeadScale& S, int nc, uint32_t taddr_a, const float* bias_a,
                                                        float* hout_a, bool active, int img, int a, int pos) {
    uint32_t rb[5];
    tmem_ld4(taddr_a, rb);
    tmem_ld1(taddr_a + 4u, rb + 4);
    tmem_wait_ld();
    pin_after_wait<5>(rb);
    float t[5];
#pragma unroll
    for (int ch = 0; ch < 5; ++ch) {
        t[ch] = activate<LEAKY>(__uint_as_float(rb[ch]), bias_a[ch], S.slope);
        if constexpr (WRITE_HEAD) {
            if (hout_a && active) hout_a[(size_t)ch * S.plane] = t[ch];
        }
    }
    float m = __int_as_float(0xff800000), m2 = m;
    int idx = 0;
    auto consume = [&](uint32_t bits, int k) {
        const float v = activate<LEAKY>(__uint_as_float(bits), bias_a[5 + k], S.slope);
        if constexpr (WRITE_HEAD) {
            if (hout_a && active) hout_a[(size_t)(5 + k) * S.plane] = v;
        }
        const bool up = v > m;
        m2 = up ? m : fmaxf(m2, v);
        idx = up ? k : idx;
        m = fmax_nan(m, v);
    };
    int k0 = 0;
#pragma unroll 1
    for (; k0 + 16 <= nc; k0 += 16) {
        uint32_t r[16];
        tmem_ld16(taddr_a + 5u + (uint32_t)k0, r);
        tmem_wait_ld();
        pin_after_wait<16>(r);
#pragma unroll
        for (int j = 0; j < 16; ++j) consume(r[j], k0 + j);
    }
#pragma unroll 1
    for (; k0 < nc; ++k0) {
        uint32_t r;
        tmem_ld1(taddr_a + 5u + (uint32_t)k0, &r);
        tmem_wait_ld();
        pin_after_wait<1>(&r);
        consume(r, k0);
    }
    if (P.emit) {
        const int gy = pos / S.nx, gx = pos - gy * S.nx;
        finish_anchor_tmem<LEAKY>(P, S, nc, active, img, a, pos, gx, gy, t[0], t[1], t[2], t[3], t[4], m, m2, idx, taddr_a + 5u, bias_a + 5);
    }
}

// 16-bit kernel: per ring stage, the producer's hand-over of a loader-filled k-block to the loader warps (one arrival once
// the stage is free).  The loader warps skip the k-blocks of TMA-filled tiles; waiting on the stage's `empty` barrier after
// such a skip would compare parities across an unknown number of phases (a CTA whose TMA tiles precede its loader tiles
// passed the wait early and double-completed the stage's loader barrier).  These barriers complete only for loader-filled
// k-blocks, in order, and never more than one phase ahead of the loader warps.  Allocated only where it is used.
template <int S>
__device__ __forceinline__ uint64_t* xgo_bars() {
    __shared__ __align__(8) uint64_t bars[S];
    return bars;
}

// X3 = fp32-accurate products from three TF32 passes (Markidis-style operand split).  The tensor core truncates an fp32
// operand to its top 19 bits (sign, exponent, 10 mantissa bits: measured, tests/test_gpu_head.py), so with
//     x = xhi + xlo,  xhi = trunc_tf32(x),   w = whi + wlo
//     D += X * W  (= xhi * whi)   +   X * Wlo  (= xhi * wlo')   +   Xlo * W  (= xlo' * whi)
// only xlo * wlo (2^-22 relative) and the truncation of the 13-bit low parts to 11 bits (2^-22) are lost: the head tensor
// matches an fp32 convolution to fp32 accumulation accuracy.  Wlo comes from the host (rows 256 .. 511 of the weight
// tensor); Xlo is computed here: two converter warps turn every X stage that lands into its low part (an elementwise
// map, so the swizzled layout carries over) before the MMA thread may use the stage.  A stage is then X | Xlo | W | Wlo
// (96 KB for 256 output channels): the ring is two stages deep, which is enough because the kernel is bound by three
// times the tensor time, not by the X stream.
constexpr int kConvThreads = 64;           // two auxiliary warps: converters in X3 mode, X loaders for unaligned planes otherwise
constexpr int kStagesX3 = 2;

template <int NA, int NC, bool WRITE_HEAD, bool LEAKY, bool X3 = false, int DT = kDtF32>
__global__ void __launch_bounds__(kProducerThreads + 128 * NA + kConvThreads, 1)
head_decode_compact_kernel(const __grid_constant__ HeadParams P) {
    // NC == 0: the class count is a run-time value (P.nc) and the accumulator keeps all 256 columns
    constexpr bool GEN = NC == 0;
    constexpr int NPAD = GEN ? kMaxN : (NA * (NC + 5) + 15) / 16 * 16;
    const int NO = GEN ? P.nc + 5 : NC + 5, N = NA * NO;
    static_assert(NPAD <= kMaxN, "one accumulator stage holds at most 256 output channels");
    // 16-bit feature maps: the k-block, the X atom and the MMA's K differ; the stage sizes are those of fp32
    constexpr bool H = DT != kDtF32;
    static_assert(!(H && X3), "the three-pass mode is fp32 only");
    constexpr int BK = H ? kBK16 : kBK;            // channels per stage
    constexpr int AS = H ? 6 : 5, AP = 1 << AS;   // positions per X swizzle atom, and its log2
    constexpr int kAtom = H ? kAtomBytes16 : kAtomBytes;
    constexpr int kBBytes = NPAD * kBK * 4;        // = NPAD * kBK16 * 2
    constexpr int kStages = X3 ? kStagesX3 : hd::kStages;
    constexpr int kXBytes = X3 ? 2 * kABytes : kABytes;           // X (and its low part)
    constexpr int kStageBytes = kXBytes + (X3 ? 2 : 1) * kBBytes;

    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full[kStages];
    __shared__ __align__(8) uint64_t empty[kStages];
    __shared__ __align__(8) uint64_t conv[kStages];              // X3: the low part of the stage's X tile is in place;
                                                                 // else: the loader warps' copies of the X tile have landed
    __shared__ __align__(8) uint64_t tfull[2];
    __shared__ __align__(8) uint64_t tempty[2];
    __shared__ uint32_t tmem_base_s;
    constexpr int kBiasPitch = ((GEN ? kMaxN / NA : NC + 5) + 3) / 4 * 4;
    __shared__ __align__(16) float bias_s[YOLO_B200_MAX_SCALES][NA][kBiasPitch];

    const int warp = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
    for (int i = threadIdx.x; i < P.n_scales * N; i += blockDim.x) {
        const int k = i / N, o = i - k * N;
        bias_s[k][o / NO][o % NO] = P.sc[k].bias[o];
    }
    // the swizzle atoms are 1024 bytes: align the ring in the shared window
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); mbar_init(&conv[s], X3 ? kConvThreads / 32 : kConvThreads); }
#pragma unroll
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 4 * NA); }
        if constexpr (H) {
#pragma unroll
            for (int s = 0; s < kStages; ++s) mbar_init(&xgo_bars<kStages>()[s], 1);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tmem_base_s)), "r"((uint32_t)kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    // One launch covers every scale: global tile index -> (scale, image, first position).  The scales are ordered
    // heaviest (largest c_in) first and the tiles are dealt round-robin, so every CTA gets the same mix and the last
    // wave consists of the cheapest tiles.
    auto locate = [&](int tile, int& k, int& img, int& p0, int& np) {
        k = 0;
#pragma unroll
        for (int j = 1; j < YOLO_B200_MAX_SCALES; ++j)
            if (j < P.n_scales && tile >= P.sc[j].first_tile) k = j;
        const int local = tile - P.sc[k].first_tile;
        img = local / P.sc[k].tiles_per_img;
        p0 = (local - img * P.sc[k].tiles_per_img) * kM;
        np = min(kM, P.sc[k].plane - p0);
    };

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            for (int k = 0; k < P.n_scales; ++k) {
                if (!P.sc[k].manual) tma_prefetch_desc(&P.sc[k].tmap_x);
                if (P.sc[k].use_x3) tma_prefetch_desc(&P.sc[k].tmap_x3);
                tma_prefetch_desc(&P.sc[k].tmap_w);
            }
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
                int k, img, p0, np;
                locate(tile, k, img, p0, np);
                const HeadScale& S = P.sc[k];
                const int atoms = (np + AP - 1) >> AS;         // boxes that start inside the plane; the rest stays stale
                // One 3-D box brings all four atoms of a k-block (a TMA instruction costs the producer ~70 ns whatever its
                // size -- profiles/r01_l_*: four boxes per k-block made the issue rate the bound).  The 3-D view only holds
                // the plane's complete 32-position atoms, so the tile with the ragged last atom uses 2-D boxes.
                // (16-bit: two atoms of 64 positions, the same rules.)
                const bool one_box = S.use_x3 && (np & (AP - 1)) == 0;
                for (int kb = 0; kb < S.kblocks; ++kb, ++it) {
                    const int st = (int)(it % kStages);
                    mbar_wait(&empty[st], ((it / kStages) & 1u) ^ 1u, P.overflow, 1);
                    const uint32_t a_s = ring + (uint32_t)st * kStageBytes;
                    // profiling modes (bits 1, 2 of skip_epilogue): fetch W / X only during the first trip round the ring
                    const bool load_w = !(P.skip_epilogue & 2) || it < (uint32_t)kStages;
                    const bool load_x = (!(P.skip_epilogue & 4) || it < (uint32_t)kStages) && !S.manual;   // manual: the loader warps
                    mbar_expect_tx(&full[st], (uint32_t)((load_x ? (one_box || P.nhwc ? kABytes : atoms * kAtom) : 0) +
                                                         (load_w ? (X3 ? 2 : 1) * kBBytes : 0)));
                    if (load_x) {
                        if (P.nhwc)       // [BK channels = 128 bytes] x [128 positions] of one image; rows past the plane zero
                            tma_tile3_g2s(a_s, &S.tmap_x, kb * BK, p0, img, &full[st]);
                        else if (one_box)
                            tma_tile3_g2s(a_s, &S.tmap_x3, 0, img * S.c_in + kb * BK, p0 >> AS, &full[st]);
                        else
                            for (int j = 0; j < atoms; ++j)
                                tma_tile_g2s(a_s + (uint32_t)j * kAtom, &S.tmap_x, p0 + AP * j, img * S.c_in + kb * BK, &full[st]);
                    }
                    if constexpr (H) {
                        if (S.manual) mbar_arrive(&xgo_bars<kStages>()[st]);   // the loader warps may fill this stage
                    }
                    if (load_w) {
                        tma_tile_g2s(a_s + kXBytes, &S.tmap_w, kb * BK, 0, &full[st]);
                        if constexpr (X3) tma_tile_g2s(a_s + kXBytes + kBBytes, &S.tmap_w, kb * kBK, kMaxN, &full[st]);   // rows 256..: w - trunc(w)
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t idesc_mn = H ? instr_desc_f16(kM, NPAD, DT == kDtBF16) : instr_desc_tf32(kM, NPAD);
            // channels_last X: A is K-major (bit 15 clear) in the SWIZZLE_128B layout of B -- 8-position groups 1 KB apart
            // (SBO), each MMA's K step 32 bytes further along the 128-byte row (8 tf32 or 16 16-bit channels)
            const bool nhwc = P.nhwc != 0;
            const uint32_t idesc = nhwc ? idesc_mn & ~(1u << 15) : idesc_mn;
            const uint32_t a_step = nhwc ? 32u : (H ? 2048u : 1024u);
            const uint64_t a_fixed = nhwc ? smem_desc(0, 16u, 1024u, kSw128)
                                          : H ? smem_desc(0, kAtomBytes16, 1024u, kSw128) : smem_desc(0, kAtomBytes, 512u, kSw128Base32);
            uint32_t it = 0, xparity = 0;
            int tl = 0;
            for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tl) {
                int k, img, p0, np;
                locate(tile, k, img, p0, np);
                const int kblocks = P.sc[k].kblocks;
                const bool manual = !X3 && P.sc[k].manual;
                const int acc = tl & 1;
                mbar_wait(&tempty[acc], (((uint32_t)tl >> 1) & 1u) ^ 1u, P.overflow, 2);   // epilogue drained this stage
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * NPAD;
                for (int kb = 0; kb < kblocks; ++kb, ++it) {
                    const int st = (int)(it % kStages);
                    mbar_wait(X3 ? &conv[st] : &full[st], (it / kStages) & 1u, P.overflow, 3);
                    if (manual) {
                        // conv[st] completes a phase only for tiles the loader warps filled: its parity is tracked per stage
                        mbar_wait(&conv[st], (xparity >> st) & 1u, P.overflow, 6);
                        xparity ^= 1u << st;
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // LDGSTS writes -> tensor-core reads
                    }
                    tc_fence_after();
                    if (P.skip_epilogue & 8) { mbar_arrive(&empty[st]); continue; }   // profiling: the stream without the tensor core
                    const uint32_t a_s = ring + (uint32_t)st * kStageBytes, b_s = a_s + kXBytes;
                    if constexpr (H) {
#pragma unroll
                        for (int kk = 0; kk < kBK16 / 16; ++kk) {
                            // A: MN-major SWIZZLE_128B: an atom is 64 positions (one 128-byte row per channel) x 8 channels;
                            //    the tile's two 64-position atoms are kAtomBytes16 apart (LBO), 8-channel groups 1 KB apart
                            //    (SBO), so this instruction's 16 channels start 2 KB after the previous one's
                            // B: K-major, as in fp32: 8-row groups 1 KB apart (SBO); 16 channels = 32 bytes inside the row
                            const uint64_t ad = smem_desc_at(a_fixed, a_s + (uint32_t)kk * a_step);
                            const uint64_t bd = smem_desc(b_s + (uint32_t)kk * 32u, 16u, 1024u, kSw128);
                            umma_f16(d_tmem, ad, bd, idesc, (kb | kk) != 0);
                        }
                    } else {
#pragma unroll
                    for (int kk = 0; kk < kBK / 8; ++kk) {
                        // A: MN-major, 32-byte-base swizzle: 4 atoms of 32 positions kAtomBytes apart (LBO); one channel is one
                        //    128-byte row, a swizzle atom is 4 rows, so this instruction's 8 channels are two atoms 512 bytes
                        //    apart (SBO) and the next instruction starts 1 KB further
                        // B: K-major, 8-row groups 1 KB apart (SBO); 8 channels = 32 bytes inside the 128-byte row
                        const uint64_t ad = smem_desc_at(a_fixed, a_s + (uint32_t)kk * a_step);
                        const uint64_t bd = smem_desc(b_s + (uint32_t)kk * 32u, 16u, 1024u, kSw128);
                        umma_tf32(d_tmem, ad, bd, idesc, (kb | kk) != 0);
                        if constexpr (X3) {
                            const uint64_t ad_lo = smem_desc_at(a_fixed, a_s + kABytes + (uint32_t)kk * a_step);
                            const uint64_t bd_lo = smem_desc(b_s + kBBytes + (uint32_t)kk * 32u, 16u, 1024u, kSw128);
                            umma_tf32(d_tmem, ad, bd_lo, idesc, true);
                            umma_tf32(d_tmem, ad_lo, bd, idesc, true);
                        }
                    }
                    }
                    umma_commit(&empty[st]);          // the stage is free once these MMAs have read it
                }
                if (P.skip_epilogue & 8) mbar_arrive(&tfull[acc]);
                else umma_commit(&tfull[acc]);        // accumulator complete
            }
        }
    } else if (!X3 && warp >= 2 + 4 * NA) {
        // ===== loader warps: the X tiles of scales whose planes have no 16-byte pitch (19x19, 13x13) =====
        // TMA cannot describe such a map (the row pitch of a tensor map is a multiple of 16 bytes, and a tile load whose
        // innermost coordinate is not 16-byte aligned faults), so these 64 threads fill the stage themselves with 4-byte
        // asynchronous copies (LDGSTS: no registers, so four stages of copies are in flight like the TMA ring's), writing
        // the layout TMA's SWIZZLE_128B_ATOM_32B gives: atom a = position / 32 (4 KB), channel row r at r * 128 bytes, the
        // 32-byte chunk (position / 8) % 4 XOR-ed with r % 4.  Lanes run along positions: coalesced 128-byte reads.
        const int lt = (int)threadIdx.x - (kProducerThreads + 128 * NA);
        uint32_t it = 0;
        uint32_t gparity = 0;                         // 16-bit: phase parity of each stage's hand-over barrier
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
            int k, img, p0, np;
            locate(tile, k, img, p0, np);
            const HeadScale& S = P.sc[k];
            if (!S.manual) { it += (uint32_t)S.kblocks; continue; }
            if constexpr (H) {
                // 16-bit (planes with 4-byte aligned rows, plane % 8 != 0): TMA's SWIZZLE_128B layout -- atom = position / 64
                // (8 KB), channel row r at r * 128 bytes, the 16-byte chunk (position / 8) % 8 XOR-ed with r % 8.
                //   plane % 4 == 0: 8-byte copies of 4 positions; lane = 4-position group (256 contiguous bytes per warp and
                //                   row), warp w of the two takes channel rows 32 w .. 32 w + 31 of every k-block;
                //   plane % 4 == 2: 4-byte copies of 2 positions; a thread owns positions 2 lt, 2 lt + 1 in all 64 rows.
                // The row-dependent parts of the offset are compile-time after unrolling (r % 8 == i % 8).
                const uint16_t* tile_src = reinterpret_cast<const uint16_t*>(S.x) + (size_t)img * S.c_in * S.plane + p0;
                const bool wide = (S.plane & 3) == 0;
                const int p = wide ? 4 * (lt & 31) : 2 * lt;
                const int r0 = wide ? 32 * (lt >> 5) : 0;
                const bool v = p < np;
                const uint32_t d = (uint32_t)((p >> 6) * kAtomBytes16 + (p & 7) * 2 + r0 * 128);
                const int c = (p >> 3) & 7;
                uint32_t xo[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) xo[q] = d + (uint32_t)((c ^ q) << 4);
                for (int kb = 0; kb < S.kblocks; ++kb, ++it) {
                    const int st = (int)(it % kStages);
                    mbar_wait(&xgo_bars<kStages>()[st], (gparity >> st) & 1u, P.overflow, 7);   // the stage is free
                    gparity ^= 1u << st;
                    const uint32_t a_s = ring + (uint32_t)st * kStageBytes;
                    const uint16_t* src = tile_src + (size_t)(kb * kBK16 + r0) * S.plane + p;
                    if (v) {
                        if (wide) {
#pragma unroll
                            for (int i = 0; i < 32; ++i, src += S.plane) cp_async8(a_s + (uint32_t)(i * 128) + xo[i & 7], src);
                        } else {
#pragma unroll
                            for (int i = 0; i < kBK16; ++i, src += S.plane) cp_async4(a_s + (uint32_t)(i * 128) + xo[i & 7], src);
                        }
                    }
                    cp_async_arrive(&conv[st]);
                }
            } else {
            // a thread owns two positions of the tile, lt and lt + 64, for all 32 channel rows of every k-block: the
            // position-dependent parts of the shared-memory offset are computed once per tile, the row-dependent ones are
            // compile-time after unrolling, and the source pointers advance by one plane per row
            const int pa = lt, pb = lt + kConvThreads;
            const bool va = pa < np, vb = pb < np;
            const uint32_t da = (uint32_t)((pa >> 5) * kAtomBytes + (pa & 7) * 4), db = (uint32_t)((pb >> 5) * kAtomBytes + (pb & 7) * 4);
            const int ca = (pa >> 3) & 3, cb = (pb >> 3) & 3;
            uint32_t xa[4], xb_[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) { xa[q] = da + (uint32_t)((ca ^ q) << 5); xb_[q] = db + (uint32_t)((cb ^ q) << 5); }
            const float* tile_src = S.x + (size_t)img * S.c_in * S.plane + p0;
            for (int kb = 0; kb < S.kblocks; ++kb, ++it) {
                const int st = (int)(it % kStages);
                mbar_wait(&empty[st], ((it / kStages) & 1u) ^ 1u, P.overflow, 7);
                const uint32_t a_s = ring + (uint32_t)st * kStageBytes;
                const float* src = tile_src + (size_t)(kb * kBK) * S.plane;
#pragma unroll
                for (int r = 0; r < kBK; ++r, src += S.plane) {
                    if (va) cp_async4(a_s + (uint32_t)(r * 128) + xa[r & 3], src + pa);
                    if (vb) cp_async4(a_s + (uint32_t)(r * 128) + xb_[r & 3], src + pb);
                }
                cp_async_arrive(&conv[st]);
            }
            }
        }
    } else if (X3 && warp >= 2 + 4 * NA) {
        // ===== X3: converter warps -- the low part of every X stage, in the layout the TMA gave the stage =====
        const int ct = (int)threadIdx.x - (kProducerThreads + 128 * NA);
        uint32_t it = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
            int k, img, p0, np;
            locate(tile, k, img, p0, np);
            for (int kb = 0; kb < P.sc[k].kblocks; ++kb, ++it) {
                const int st = (int)(it % kStages);
                mbar_wait(&full[st], (it / kStages) & 1u, P.overflow, 5);
                uint8_t* stage = smem_raw + (ring - smem_u32(smem_raw)) + (size_t)st * kStageBytes;
                const float4* x = reinterpret_cast<const float4*>(stage);
                float4* xlo = reinterpret_cast<float4*>(stage + kABytes);
#pragma unroll 4
                for (int i = ct; i < kABytes / 16; i += kConvThreads) {
                    const float4 v = x[i];
                    float4 l;
                    l.x = __fsub_rn(v.x, __uint_as_float(__float_as_uint(v.x) & 0xffffe000u));
                    l.y = __fsub_rn(v.y, __uint_as_float(__float_as_uint(v.y) & 0xffffe000u));
                    l.z = __fsub_rn(v.z, __uint_as_float(__float_as_uint(v.z) & 0xffffe000u));
                    l.w = __fsub_rn(v.w, __uint_as_float(__float_as_uint(v.w) & 0xffffe000u));
                    xlo[i] = l;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // generic-proxy stores -> tensor-core reads
                __syncwarp();
                if (lane == 0) mbar_arrive(&conv[st]);
            }
        }
    } else {
        // ===== epilogue warps: one warp per (TMEM lane quarter, anchor) =====
        // A warp may only touch the TMEM lanes 32 * (warp index mod 4) .. + 31; warps 2 .. 2 + 4 * NA - 1 cover every
        // (quarter, anchor) pair once.  Four warps per anchor instead of four per tile: the per-anchor atomic round trip of the
        // candidate emission and the TMEM load latency overlap across the NA warps that share a scheduler.
        const int q = warp & 3;
        const int a = (warp - 2) >> 2;
        const int row = q * 32 + lane;                // TMEM lane = position inside the tile
        int tl = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++tl) {
            int k, img, p0, np;
            locate(tile, k, img, p0, np);
            const HeadScale& S = P.sc[k];
            const int acc = tl & 1;
            const bool active = row < np;
            const int pos = active ? p0 + row : p0;
            mbar_wait<true>(&tfull[acc], ((uint32_t)tl >> 1) & 1u, P.overflow, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * NPAD;
            float* hout_a = S.head_out ? S.head_out + ((size_t)img * N + (size_t)a * NO) * S.plane + pos : nullptr;
            if (!(P.skip_epilogue & 1)) {
                if constexpr (GEN)
                    epilogue_anchor_generic<WRITE_HEAD, LEAKY>(P, S, P.nc, taddr + (uint32_t)(a * NO), bias_s[k][a], hout_a, active, img, a, pos);
                else
                    epilogue_anchor<NC, WRITE_HEAD, LEAKY>(P, S, taddr + (uint32_t)(a * NO), bias_s[k][a], hout_a, active, img, a, pos);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTmemCols) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): two CTAs on neighbouring SMs share one 256-position tile.  Each CTA stages
// its own 128 positions of X and only HALF of the W rows; the pair's tensor cores read both halves.  A ring stage is
// 32 KB instead of 48 KB, so six stages fit and 96 KB instead of 64 KB of X are in flight per SM -- the single-CTA
// kernel is bound by exactly that (X streams at bytes-in-flight / ~2 us TMA latency, profiles/r01_k_fused_head_v2.txt).
//   * full[] lives in the leader (rank 0): both CTAs' TMA loads complete_tx on it, the leader arms it with the pair's bytes
//   * empty[] and tfull[] are per CTA: the leader's tcgen05.commit multicasts its arrival to both
//   * tempty[] lives in the leader: the epilogue warps of both CTAs arrive on it (remote arrive from rank 1)
constexpr int kStages2 = 6;
constexpr uint32_t kPeerMask = 0xFEFFFFFFu;     // shared::cluster address of the same variable in the pair's leader CTA

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_tile_g2s_2cta(uint32_t dst, const CUtensorMap* map, int x, int y, uint32_t leader_bar) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(leader_bar), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_tile3_g2s_2cta(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, uint32_t leader_bar) {
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void umma_tf32_2cta(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"((uint32_t)accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {        // arrives on `bar` in both CTAs of the pair
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar_addr) : "memory");
}

template <int NA, int NC, bool WRITE_HEAD, bool LEAKY>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kProducerThreads + 128 * NA, 1)
head_decode_compact_2cta_kernel(const __grid_constant__ HeadParams P) {
    constexpr int NO = NC + 5, N = NA * NO, NPAD = (N + 15) / 16 * 16;
    static_assert(NPAD <= kMaxN && NPAD % 16 == 0, "one accumulator stage holds at most 256 output channels");
    constexpr int kHalfN = NPAD / 2;                     // W rows staged by each CTA
    constexpr int kBBytes = kHalfN * kBK * 4;
    constexpr int kStageBytes = kABytes + kBBytes;
    static_assert(kStageBytes % 1024 == 0, "stages must keep the 1 KB swizzle-atom alignment");

    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full[kStages2];
    __shared__ __align__(8) uint64_t empty[kStages2];
    __shared__ __align__(8) uint64_t tfull[2];
    __shared__ __align__(8) uint64_t tempty[2];
    __shared__ uint32_t tmem_base_s;
    constexpr int kBiasPitch = (NO + 3) / 4 * 4;
    __shared__ __align__(16) float bias_s[NA][kBiasPitch];

    const HeadScale& S = P.sc[P.pair_scale];
    const int warp = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = (int)blockIdx.x >> 1, n_pairs = (int)gridDim.x >> 1;
    const int tiles_per_img = (S.plane + 2 * kM - 1) / (2 * kM);
    const int n_tiles = P.batch * tiles_per_img;
    for (int i = threadIdx.x; i < N; i += blockDim.x) bias_s[i / NO][i % NO] = S.bias[i];
    const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;

    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages2; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
#pragma unroll
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], 2 * 4 * NA); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&tmem_base_s)), "r"((uint32_t)kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // the peer's barriers exist before anybody signals them
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    // this CTA's half of pair tile `tile`
    auto locate = [&](int tile, int& img, int& my_p0, int& my_np, int& pair_bytes) {
        img = tile / tiles_per_img;
        const int p0 = (tile - img * tiles_per_img) * (2 * kM);
        const int np = min(2 * kM, S.plane - p0);
        const int np0 = min(kM, np), np1 = np - np0;
        my_p0 = p0 + (int)rank * kM;
        my_np = rank ? np1 : np0;
        auto x_bytes = [&](int n) {   // what this half's producer will request: one 3-D box (always 16 KB) or 2-D boxes per atom
            const bool one_box = S.use_x3 && n > 0 && (n == kM || (n & 31) == 0);
            return one_box ? kABytes : ((n + 31) >> 5) * kAtomBytes;
        };
        pair_bytes = x_bytes(np0) + x_bytes(np1) + 2 * kBBytes;
    };

    if (warp == 0) {
        // ===== TMA producer (both CTAs; completion is counted on the leader's barrier) =====
        if (lane == 0) {
            tma_prefetch_desc(&S.tmap_x);
            tma_prefetch_desc(&S.tmap_x3);
            tma_prefetch_desc(&S.tmap_w2);
            uint32_t it = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs) {
                int img, my_p0, my_np, pair_bytes;
                locate(tile, img, my_p0, my_np, pair_bytes);
                const int atoms = (my_np + 31) >> 5;
                const bool one_box = S.use_x3 && my_np > 0 && (my_np == kM || (my_np & 31) == 0);
                for (int kb = 0; kb < S.kblocks; ++kb, ++it) {
                    const int st = (int)(it % kStages2);
                    mbar_wait(&empty[st], ((it / kStages2) & 1u) ^ 1u, P.overflow, 1);
                    const uint32_t a_s = ring + (uint32_t)st * kStageBytes;
                    const uint32_t leader_full = smem_u32(&full[st]) & kPeerMask;
                    if (rank == 0) mbar_expect_tx(&full[st], (uint32_t)pair_bytes);
                    if (one_box)
                        tma_tile3_g2s_2cta(a_s, &S.tmap_x3, 0, img * S.c_in + kb * kBK, my_p0 >> 5, leader_full);
                    else
                        for (int j = 0; j < atoms; ++j)
                            tma_tile_g2s_2cta(a_s + (uint32_t)j * kAtomBytes, &S.tmap_x, my_p0 + 32 * j, img * S.c_in + kb * kBK, leader_full);
                    tma_tile_g2s_2cta(a_s + kABytes, &S.tmap_w2, kb * kBK, (int)rank * kHalfN, leader_full);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the leader CTA drives both tensor cores =====
        if (lane == 0 && rank == 0) {
            constexpr uint32_t idesc = instr_desc_tf32(2 * kM, NPAD);
            uint32_t it = 0;
            int tl = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs, ++tl) {
                const int acc = tl & 1;
                mbar_wait(&tempty[acc], (((uint32_t)tl >> 1) & 1u) ^ 1u, P.overflow, 2);   // both epilogues drained this stage
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * NPAD;
                for (int kb = 0; kb < S.kblocks; ++kb, ++it) {
                    const int st = (int)(it % kStages2);
                    mbar_wait(&full[st], (it / kStages2) & 1u, P.overflow, 3);
                    tc_fence_after();
                    const uint32_t a_s = ring + (uint32_t)st * kStageBytes, b_s = a_s + kABytes;
#pragma unroll
                    for (int k = 0; k < kBK / 8; ++k) {
                        const uint64_t ad = smem_desc(a_s + (uint32_t)k * 1024u, kAtomBytes, 512u, kSw128Base32);
                        const uint64_t bd = smem_desc(b_s + (uint32_t)k * 32u, 16u, 1024u, kSw128);
                        umma_tf32_2cta(d_tmem, ad, bd, idesc, (kb | k) != 0);
                    }
                    umma_commit_2cta(&empty[st]);
                }
                umma_commit_2cta(&tfull[acc]);
            }
        }
    } else {
        // ===== epilogue warps (both CTAs, each on its own 128 TMEM lanes) =====
        const int q = warp & 3;
        const int a = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        int tl = 0;
        for (int tile = pair; tile < n_tiles; tile += n_pairs, ++tl) {
            const int acc = tl & 1;
            int img, my_p0, my_np, pair_bytes;
            locate(tile, img, my_p0, my_np, pair_bytes);
            const bool active = row < my_np;
            const int pos = active ? my_p0 + row : 0;
            mbar_wait<true>(&tfull[acc], ((uint32_t)tl >> 1) & 1u, P.overflow, 4);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * NPAD;
            float* hout_a = S.head_out ? S.head_out + ((size_t)img * N + (size_t)a * NO) * S.plane + pos : nullptr;
            if (!(P.skip_epilogue & 1))
                epilogue_anchor<NC, WRITE_HEAD, LEAKY>(P, S, taddr + (uint32_t)(a * NO), bias_s[a], hout_a, active, img, a, pos);
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(smem_u32(&tempty[acc]) & kPeerMask);
        }
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                                   // nobody leaves while the peer can still signal or read it
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)kTmemCols) : "memory");
    }
}

}  // namespace hd
}  // namespace yb

// ------------------------------------------------------------------------------------------------------------------
// Plane padding: (rows, plane) floats -> (rows, pitch), pitch % 4 == 0, so that a 19x19 / 13x13 feature map gets the
// 16-byte row pitch TMA needs.  One warp per channel plane, lanes on consecutive floats (the source rows start on
// arbitrary 4-byte boundaries), every load of a plane in flight before the first store.
namespace yb {
namespace hd {
constexpr int kPadThreads = 256;
constexpr int kPadMaxIter = 16;            // planes of up to 512 floats in one pass

__global__ void __launch_bounds__(kPadThreads)
pad_planes_kernel(const float* __restrict__ x, float* __restrict__ out, long long rows, int plane, int pitch) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * (kPadThreads / 32) + (threadIdx.x >> 5);
    const long long stride = (long long)gridDim.x * (kPadThreads / 32);
    for (long long r = warp0; r < rows; r += stride) {
        const float* src = x + r * plane;
        float* dst = out + r * pitch;
        for (int base = 0; base < pitch; base += 32 * kPadMaxIter) {
            float v[kPadMaxIter];
#pragma unroll
            for (int k = 0; k < kPadMaxIter; ++k) {
                const int i = base + 32 * k + lane;
                v[k] = i < plane ? ldg_stream(src + i) : 0.0f;
            }
#pragma unroll
            for (int k = 0; k < kPadMaxIter; ++k) {
                const int i = base + 32 * k + lane;
                if (i < pitch) dst[i] = v[k];
            }
        }
    }
}

// The same for 2-byte elements (fp16 / bf16 feature maps), pitch % 8 == 0: gives planes of any size -- odd ones above all,
// whose rows the kernel's loader warps cannot copy in aligned pieces -- the 16-byte row pitch TMA needs.
__global__ void __launch_bounds__(kPadThreads)
pad_planes16_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ out, long long rows, int plane, int pitch) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = (long long)blockIdx.x * (kPadThreads / 32) + (threadIdx.x >> 5);
    const long long stride = (long long)gridDim.x * (kPadThreads / 32);
    for (long long r = warp0; r < rows; r += stride) {
        const uint16_t* src = x + r * plane;
        uint16_t* dst = out + r * pitch;
        for (int base = 0; base < pitch; base += 32 * kPadMaxIter) {
            unsigned short v[kPadMaxIter];
#pragma unroll
            for (int k = 0; k < kPadMaxIter; ++k) {
                const int i = base + 32 * k + lane;
                v[k] = i < plane ? ldg_stream_b16(src + i) : (unsigned short)0;
            }
#pragma unroll
            for (int k = 0; k < kPadMaxIter; ++k) {
                const int i = base + 32 * k + lane;
                if (i < pitch) dst[i] = v[k];
            }
        }
    }
}
}  // namespace hd
}  // namespace yb

// ================================================================================================
// host side
// ================================================================================================
using namespace yb;

extern "C" int yolo_b200_pad_planes(const float* x, float* out, long long rows, int plane, int pitch, yolo_b200_stream_t stream) {
    if (rows > 0 && (!x || !out)) return YOLO_B200_E_NULL;
    if (rows < 0 || plane < 1 || pitch < plane || pitch % 4 != 0) return YOLO_B200_E_RANGE;
    if (((uintptr_t)x & 3u) || ((uintptr_t)out & 15u)) return YOLO_B200_E_ALIGN;
    if (rows == 0) return 0;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (rows + hd::kPadThreads / 32 - 1) / (hd::kPadThreads / 32);
    const int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
    hd::pad_planes_kernel<<<grid, hd::kPadThreads, 0, stream>>>(x, out, rows, plane, pitch);
    return (int)cudaGetLastError();
}

extern "C" int yolo_b200_pad_planes_16(const void* x, void* out, long long rows, int plane, int pitch, yolo_b200_stream_t stream) {
    if (rows > 0 && (!x || !out)) return YOLO_B200_E_NULL;
    if (rows < 0 || plane < 1 || pitch < plane || pitch % 8 != 0) return YOLO_B200_E_RANGE;
    if (((uintptr_t)x & 1u) || ((uintptr_t)out & 15u)) return YOLO_B200_E_ALIGN;
    if (rows == 0) return 0;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const long long want = (rows + hd::kPadThreads / 32 - 1) / (hd::kPadThreads / 32);
    const int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
    hd::pad_planes16_kernel<<<grid, hd::kPadThreads, 0, stream>>>(static_cast<const uint16_t*>(x), static_cast<uint16_t*>(out), rows,
                                                                  plane, pitch);
    return (int)cudaGetLastError();
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int encode_2d(EncodeTiledFn fn, CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t row_bytes,
                     uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swizzle,
                     CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_FLOAT32) {
    const cuuint64_t gdim[2] = {inner, outer};
    const cuuint64_t gstride[1] = {row_bytes};
    const cuuint32_t box[2] = {box_inner, box_outer};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(map, dtype, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, promo,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : YOLO_B200_E_RANGE;
}

typedef void (*HeadKernel)(const hd::HeadParams);

// the (anchors per scale, classes) pairs the epilogue is instantiated for, each with / without head_out stores and LeakyReLU
template <int NA, int NC, int DT>
static HeadKernel pick_variant16(bool write_head, bool leaky) {
    return write_head ? (leaky ? hd::head_decode_compact_kernel<NA, NC, true, true, false, DT> : hd::head_decode_compact_kernel<NA, NC, true, false, false, DT>)
                      : (leaky ? hd::head_decode_compact_kernel<NA, NC, false, true, false, DT> : hd::head_decode_compact_kernel<NA, NC, false, false, false, DT>);
}
template <int NA, int NC>
static HeadKernel pick_variant(bool write_head, bool leaky, bool pair, bool x3 = false, int dt = hd::kDtF32) {
    // 16-bit feature maps: the one-pass single-CTA kernel only
    if (dt == hd::kDtF16) return pair || x3 ? nullptr : pick_variant16<NA, NC, hd::kDtF16>(write_head, leaky);
    if (dt == hd::kDtBF16) return pair || x3 ? nullptr : pick_variant16<NA, NC, hd::kDtBF16>(write_head, leaky);
    if (x3) {
        if constexpr (NC == 80 || NC == 0) {
            return write_head ? (leaky ? hd::head_decode_compact_kernel<NA, NC, true, true, true> : hd::head_decode_compact_kernel<NA, NC, true, false, true>)
                              : (leaky ? hd::head_decode_compact_kernel<NA, NC, false, true, true> : hd::head_decode_compact_kernel<NA, NC, false, false, true>);
        } else {
            return nullptr;
        }
    }
    if (pair) {
        if constexpr (NA == 3 && NC == 80) {
            return write_head ? (leaky ? hd::head_decode_compact_2cta_kernel<NA, NC, true, true> : hd::head_decode_compact_2cta_kernel<NA, NC, true, false>)
                              : (leaky ? hd::head_decode_compact_2cta_kernel<NA, NC, false, true> : hd::head_decode_compact_2cta_kernel<NA, NC, false, false>);
        } else {
            return nullptr;
        }
    }
    return write_head ? (leaky ? hd::head_decode_compact_kernel<NA, NC, true, true> : hd::head_decode_compact_kernel<NA, NC, true, false>)
                      : (leaky ? hd::head_decode_compact_kernel<NA, NC, false, true> : hd::head_decode_compact_kernel<NA, NC, false, false>);
}
static HeadKernel head_kernel_for(int na, int nc, bool write_head, bool leaky, bool pair, bool x3 = false, int dt = hd::kDtF32) {
    if (x3) {     // three-pass mode: the 80-class epilogue or the run-time class loop, both over all 256 accumulator columns
        if (na == 3 && nc == 80) return pick_variant<3, 80>(write_head, leaky, false, true);
        if (na == 3 && nc >= 1 && na * (nc + 5) <= hd::kMaxN) return pick_variant<3, 0>(write_head, leaky, false, true);
        return nullptr;
    }
    if (na == 3 && nc == 80) return pick_variant<3, 80>(write_head, leaky, pair, false, dt);     // COCO
    if (na == 3 && nc == 20) return pick_variant<3, 20>(write_head, leaky, pair, false, dt);     // VOC
    if (na == 3 && nc == 1) return pick_variant<3, 1>(write_head, leaky, pair, false, dt);
    if (na == 3 && nc >= 2 && na * (nc + 5) <= hd::kMaxN && !pair) return pick_variant<3, 0>(write_head, leaky, false, false, dt);   // any other class count
    return nullptr;
}
// output-channel rows the kernel's accumulator / W tile holds for (na, nc)
static int head_npad(int na, int nc) {
    const bool specialised = na == 3 && (nc == 80 || nc == 20 || nc == 1);
    return specialised ? (na * (nc + 5) + 15) / 16 * 16 : hd::kMaxN;
}

// element type of X and W named by the flags: fp32, fp16, bf16, or -1 for both 16-bit bits
static int head_dtype(int flags) {
    const int h = flags & (YOLO_B200_HEAD_F16 | YOLO_B200_HEAD_BF16);
    return h == 0 ? hd::kDtF32 : h == YOLO_B200_HEAD_F16 ? hd::kDtF16 : h == YOLO_B200_HEAD_BF16 ? hd::kDtBF16 : -1;
}

extern "C" int yolo_b200_head_supported_ex(int c_in, int ny, int nx, int x_row_pitch, int na, int n_classes, int flags) {
    const int dt = head_dtype(flags);
    if (flags & YOLO_B200_HEAD_NHWC) {
        // channels_last X: one tensor-map box per k-block whatever the plane, no row pitch; not the CTA-pair kernel
        if (dt < 0 || x_row_pitch != 0 || (flags & YOLO_B200_HEAD_CTA_PAIR)) return 0;
        if (dt != hd::kDtF32 && (flags & YOLO_B200_HEAD_FP32X3)) return 0;
        const int bk = dt != hd::kDtF32 ? hd::kBK16 : hd::kBK;
        if (c_in < bk || c_in % bk != 0 || ny < 1 || nx < 1) return 0;
        return head_kernel_for(na, n_classes, false, false, false, false, dt) != nullptr ? 1 : 0;
    }
    if (dt != hd::kDtF32) {
        // 16-bit: one-pass single-CTA kernel, 64-channel k-blocks, a row pitch of 8 elements (16 bytes) unless the
        // contiguous planes are even (the loader warps copy 4-byte aligned pieces; odd planes go through the padded copy)
        if (dt < 0 || (flags & (YOLO_B200_HEAD_FP32X3 | YOLO_B200_HEAD_CTA_PAIR))) return 0;
        if (c_in < hd::kBK16 || c_in % hd::kBK16 != 0 || ny < 1 || nx < 1) return 0;
        const long long plane = (long long)ny * nx, pitch = x_row_pitch ? x_row_pitch : plane;
        if (pitch < plane) return 0;
        if (pitch % 8 != 0 && (x_row_pitch != 0 || plane % 2 != 0)) return 0;
        return head_kernel_for(na, n_classes, false, false, false, false, dt) != nullptr ? 1 : 0;
    }
    if (c_in < hd::kBK || c_in % hd::kBK != 0) return 0;
    if (ny < 1 || nx < 1) return 0;
    const long long pitch = x_row_pitch ? x_row_pitch : (long long)ny * nx;
    if (pitch < (long long)ny * nx) return 0;
    if (pitch % 4 != 0) {
        // no 16-byte row pitch, so no tensor map: contiguous planes are filled in by the kernel's loader warps, which the
        // one-pass single-CTA kernel has; the three-pass mode and the CTA-pair kernel need the padded copy
        if (x_row_pitch != 0 || (flags & (YOLO_B200_HEAD_FP32X3 | YOLO_B200_HEAD_CTA_PAIR))) return 0;
    }
    return head_kernel_for(na, n_classes, false, false, false) != nullptr ? 1 : 0;
}
extern "C" int yolo_b200_head_supported(int c_in, int ny, int nx, int x_row_pitch, int na, int n_classes) {
    return yolo_b200_head_supported_ex(c_in, ny, nx, x_row_pitch, na, n_classes, 0);
}

extern "C" int yolo_b200_head_decode_compact(const yolo_b200_head* heads, int n_heads, int batch, int nc, int rows_per_img,
                                             float conf_thres, float min_wh,
                                             yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                             int32_t* count, int32_t* overflow, int flags, yolo_b200_stream_t stream) {
    if (!heads || !count || !overflow) return YOLO_B200_E_NULL;
    const bool emit = (flags & YOLO_B200_HEAD_NO_CANDIDATES) == 0;
    const bool x3 = (flags & YOLO_B200_HEAD_FP32X3) != 0;
    if (x3 && (flags & YOLO_B200_HEAD_CTA_PAIR)) return YOLO_B200_E_RANGE;
    const int dt = head_dtype(flags);
    if (dt < 0) return YOLO_B200_E_RANGE;
    const bool h16 = dt != hd::kDtF32;
    if (h16 && (flags & (YOLO_B200_HEAD_FP32X3 | YOLO_B200_HEAD_CTA_PAIR))) return YOLO_B200_E_UNSUPPORTED;
    const bool nhwc = (flags & YOLO_B200_HEAD_NHWC) != 0;
    if (nhwc && (flags & YOLO_B200_HEAD_CTA_PAIR)) return YOLO_B200_E_UNSUPPORTED;
    if (emit && (!cand_box || !cand_meta)) return YOLO_B200_E_NULL;
    if (n_heads < 1 || n_heads > YOLO_B200_MAX_SCALES || batch < 0 || nc < 1 || rows_per_img < 1 || (emit && cap_per_img < 1))
        return YOLO_B200_E_RANGE;
    if (emit && ((((uintptr_t)cand_box) | ((uintptr_t)cand_meta)) & 15u)) return YOLO_B200_E_ALIGN;
    // validate everything before the first launch
    for (int k = 0; k < n_heads; ++k) {
        const yolo_b200_head& h = heads[k];
        if (batch > 0 && (!h.x || !h.weight || !h.bias_host)) return YOLO_B200_E_NULL;
        if (h.x_row_pitch < 0) return YOLO_B200_E_RANGE;
        if (!yolo_b200_head_supported_ex(h.c_in, h.scale.ny, h.scale.nx, h.x_row_pitch, h.scale.na, nc, flags)) return YOLO_B200_E_UNSUPPORTED;
        if (h.negative_slope < 0.0f || h.negative_slope > 1.0f) return YOLO_B200_E_RANGE;
        if ((((uintptr_t)h.x) | ((uintptr_t)h.weight)) & 15u) return YOLO_B200_E_ALIGN;
        if (h.head_out && ((uintptr_t)h.head_out & 3u)) return YOLO_B200_E_ALIGN;
        if (h.scale.row_off < 0 || (long long)h.scale.row_off + (long long)h.scale.na * h.scale.ny * h.scale.nx > rows_per_img)
            return YOLO_B200_E_RANGE;
        if ((long long)batch * h.c_in > 0x7fffffffLL) return YOLO_B200_E_RANGE;
    }
    cudaError_t e;
    if (!(flags & YOLO_B200_HEAD_ACCUMULATE)) {
        if (overflow == count + batch) e = cudaMemsetAsync(count, 0, sizeof(int32_t) * (batch + 1), stream);
        else {
            e = batch > 0 ? cudaMemsetAsync(count, 0, sizeof(int32_t) * batch, stream) : cudaSuccess;
            if (e == cudaSuccess) e = cudaMemsetAsync(overflow, 0, sizeof(int32_t), stream);
        }
        if (e != cudaSuccess) return (int)e;
    }
    if (batch == 0) return 0;

    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if ((e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres)) != cudaSuccess) return (int)e;
    if (!fn || qres != cudaDriverEntryPointSuccess) return YOLO_B200_E_RANGE;
    EncodeTiledFn encode = (EncodeTiledFn)fn;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);

    // L2 promotion 64 B .. 256 B and the plain 128-byte swizzle make no measurable difference for the X stream
    // (profiles/r01_l_tma_box_rows_experiment.txt); MN-major tf32 requires the 32-byte-atom swizzle.
    // 16-bit: plain SWIZZLE_128B, the MN-major layout kind::f16 reads; 64-position atoms
    const CUtensorMapSwizzle x_swizzle = h16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    const CUtensorMapDataType x_type = dt == hd::kDtF16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                                      : dt == hd::kDtBF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    const uint64_t esz = h16 ? 2 : 4;
    const int bk = h16 ? hd::kBK16 : hd::kBK, ap = h16 ? 64 : 32;
    const CUtensorMapL2promotion x_promo = CU_TENSOR_MAP_L2_PROMOTION_L2_128B;
    const int no = nc + 5;

    // Heads that share the anchor count run in ONE launch (the kernel is instantiated per (anchors, classes)); inside a
    // launch the scales are ordered heaviest first.  Reference models use 3 anchors on every scale.
    bool done[YOLO_B200_MAX_SCALES] = {false, false, false, false};
    for (int first = 0; first < n_heads; ++first) {
        if (done[first]) continue;
        const int na = heads[first].scale.na, n = na * no, npad = x3 ? hd::kMaxN : head_npad(na, nc);
        int order[YOLO_B200_MAX_SCALES], cnt = 0;
        for (int k = first; k < n_heads; ++k)
            if (!done[k] && heads[k].scale.na == na) { order[cnt++] = k; done[k] = true; }
        for (int i = 0; i < cnt; ++i)
            for (int j = i + 1; j < cnt; ++j)
                if (heads[order[j]].c_in > heads[order[i]].c_in) { const int t = order[i]; order[i] = order[j]; order[j] = t; }

        hd::HeadParams P{};
        long long tiles = 0;
        for (int i = 0; i < cnt; ++i) {
            const yolo_b200_head& h = heads[order[i]];
            hd::HeadScale& S = P.sc[i];
            const int plane = h.scale.ny * h.scale.nx;
            const uint64_t pitch = h.x_row_pitch ? (uint64_t)h.x_row_pitch : (uint64_t)plane;      // elements between channel planes
            int rc;
            S.manual = !nhwc && pitch % (16 / esz) != 0 ? 1 : 0;   // (validated above: contiguous planes, one-pass single-CTA kernel)
            S.x = h.x;
            if (nhwc) {
                // channels_last: (c_in, plane, batch), box = one k-block of channels (128 bytes) x 128 positions x 1 image,
                // positions past the plane zero-filled; c_in * esz is a multiple of 128 bytes
                const cuuint64_t gdim[3] = {(cuuint64_t)h.c_in, (cuuint64_t)plane, (cuuint64_t)batch};
                const cuuint64_t gstride[2] = {(cuuint64_t)h.c_in * esz, (cuuint64_t)plane * h.c_in * esz};
                const cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)hd::kM, 1};
                const cuuint32_t estr[3] = {1, 1, 1};
                if (encode(&S.tmap_x, x_type, 3, const_cast<float*>(h.x), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                           CU_TENSOR_MAP_SWIZZLE_128B, x_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                    return YOLO_B200_E_RANGE;
            } else if (!S.manual &&
                (rc = encode_2d(encode, &S.tmap_x, h.x, (uint64_t)plane, (uint64_t)batch * h.c_in, pitch * esz, ap, bk, x_swizzle, x_promo, x_type)))
                return rc;
            // (three-pass mode: the tensor holds 512 rows, the low parts of the weights behind the weights)
            if ((rc = encode_2d(encode, &S.tmap_w, h.weight, (uint64_t)h.c_in, (uint64_t)(x3 ? 2 * npad : npad), (uint64_t)h.c_in * esz, bk,
                                (uint32_t)npad, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, x_type)))
                return rc;
            if (!h16 && (rc = encode_2d(encode, &S.tmap_w2, h.weight, (uint64_t)h.c_in, (uint64_t)npad, (uint64_t)h.c_in * 4, hd::kBK,
                                        (uint32_t)npad / 2, CU_TENSOR_MAP_SWIZZLE_128B)))
                return rc;
            // 3-D view over the complete atoms (32 positions, 16-bit: 64) of every row; rows are pitch elements apart, atoms
            // 128 bytes; the box is the tile's four (16-bit: two) atoms
            S.use_x3 = 0;
            if (!nhwc && plane >= ap && !S.manual) {
                const cuuint64_t gdim[3] = {(cuuint64_t)ap, (cuuint64_t)batch * h.c_in, (cuuint64_t)(plane / ap)};
                const cuuint64_t gstride[2] = {(cuuint64_t)pitch * esz, 128};
                const cuuint32_t box[3] = {(cuuint32_t)ap, (cuuint32_t)bk, (cuuint32_t)(hd::kM / ap)};
                const cuuint32_t estr[3] = {1, 1, 1};
                const CUresult r3 = encode(&S.tmap_x3, x_type, 3, const_cast<float*>(h.x), gdim, gstride, box, estr,
                                           CU_TENSOR_MAP_INTERLEAVE_NONE, x_swizzle, x_promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
                S.use_x3 = r3 == CUDA_SUCCESS ? 1 : 0;        // a driver that rejects the view leaves the 2-D boxes
            }
            for (int o = 0; o < hd::kMaxN; ++o) S.bias[o] = o < n ? h.bias_host[o] : 0.0f;
            S.slope = h.negative_slope;
            S.c_in = h.c_in; S.kblocks = h.c_in / bk;
            S.ny = h.scale.ny; S.nx = h.scale.nx; S.plane = plane; S.row_off = h.scale.row_off;
            S.tiles_per_img = (plane + hd::kM - 1) / hd::kM;
            S.first_tile = (int)tiles;
            tiles += (long long)batch * S.tiles_per_img;
            if (tiles > 0x7fffffffLL) return YOLO_B200_E_RANGE;
            S.stride = h.scale.stride;
            for (int a = 0; a < YOLO_B200_MAX_ANCHORS; ++a) { S.av[a][0] = h.scale.anchor_vec[a][0]; S.av[a][1] = h.scale.anchor_vec[a][1]; }
            S.head_out = h.head_out;
        }
        P.n_scales = cnt; P.batch = batch; P.n_tiles = (int)tiles; P.nc = nc;
        P.conf = conf_thres; P.min_wh = min_wh;
        P.cand_box = cand_box; P.cand_meta = cand_meta; P.cap = cap_per_img; P.count = count; P.overflow = overflow;
        P.emit = emit ? 1 : 0;
        P.nhwc = nhwc ? 1 : 0;
        P.skip_epilogue = (flags >> 8) & 15;     // YOLO_B200_HEAD_PROFILE_* bits

        // The CTA-pair kernel is exact but measured ~5 % slower than the single-CTA kernel on B200 (profiles/r01_m_*): on
        // request only, one launch per scale
        bool write_head = false, leaky = false;
        for (int i = 0; i < cnt; ++i) {
            write_head |= heads[order[i]].head_out != nullptr;
            leaky |= heads[order[i]].negative_slope != 1.0f;
        }
        HeadKernel kern2 = (flags & YOLO_B200_HEAD_CTA_PAIR) ? head_kernel_for(na, nc, write_head, leaky, true) : nullptr;
        if (kern2) {
            const size_t smem = (size_t)hd::kStages2 * (hd::kABytes + (size_t)(npad / 2) * hd::kBK * 4) + 1024;
            if ((e = cudaFuncSetAttribute((const void*)kern2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
            for (int i = 0; i < cnt; ++i) {
                P.pair_scale = i;
                const long long pairs = (long long)batch * ((P.sc[i].plane + 2 * hd::kM - 1) / (2 * hd::kM));
                const int max_pairs = sms / 2;
                const int grid = 2 * (int)(pairs < max_pairs ? pairs : max_pairs);
                kern2<<<grid, hd::kProducerThreads + 128 * na, smem, stream>>>(P);
                if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
            }
            continue;
        }
        HeadKernel kern = head_kernel_for(na, nc, write_head, leaky, false, x3, dt);
        if (!kern) return YOLO_B200_E_UNSUPPORTED;
        const size_t smem = x3 ? (size_t)hd::kStagesX3 * 2 * (hd::kABytes + (size_t)npad * hd::kBK * 4) + 1024
                               : (size_t)hd::kStages * (hd::kABytes + (size_t)npad * hd::kBK * 4) + 1024;
        if ((e = cudaFuncSetAttribute((const void*)kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return (int)e;
        const int grid = (int)(tiles < sms ? tiles : sms);
        kern<<<grid, hd::kProducerThreads + 128 * na + hd::kConvThreads, smem, stream>>>(P);
        if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
    }
    return 0;
}
