// Decode-side kernels of the yolo_b200 hot path (sm_100a).
//
//   decode_compact_kernel      fused YOLOLayer decode + confidence filter + stream compaction
//                              (reference models/yolo_layer.py:90-99 + utils/utils.py:210-234)
//   decode_dense_kernel        API-parity decode: writes the (B, N, 5+nc) tensor model.forward returns
//                              (reference models/yolo_layer.py:57-99 + models/yolov3_spp.py:163-164)
//   compact_from_dense_kernel  the filter/compaction half of non_max_suppression on an already decoded
//                              tensor (reference utils/utils.py:210-234), fed by TMA bulk copies
//
// All three are HBM-bound streaming kernels that read each input byte at most once.  decode_compact_kernel reads the
// objectness plane whole and the box and class planes only around positions whose objectness can pass the confidence
// threshold; decode_compact_dense_kernel (selectable) and the other kernels read every byte once.
#include <cuda.h>          // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"

namespace yb {

// ------------------------------------------------------------------------------------------------
// Launch-time description of one scale, derived on the host from yolo_b200_scale.
struct ScaleDev {
    const void* head; // fp32 elements; 16-bit elements in decode_compact's F16 / BF16 modes (LDG kernels only)
    int ny, nx, na, row_off;
    int plane;        // ny*nx
    int vec;          // 4 when every (slab, channel) plane start is aligned to 4 elements (16 bytes fp32, 8 bytes 16-bit), else 1
    int n_units;      // batch*na*plane / vec   work units of this scale
    int first_block;  // first blockIdx.x that works on this scale
    int first_tile;   // TMA kernel: first tile id of this scale
    int tiles_per_slab;
    float stride;
    float av[YOLO_B200_MAX_ANCHORS][2];
};

struct DecodeParams {
    ScaleDev sc[YOLO_B200_MAX_SCALES];
    int n_scales, batch, nc, rows_per_img;
    float conf, min_wh;
    yolo_b200_box* cand_box;
    yolo_b200_meta* cand_meta;
    int cap;
    int32_t* count;
    int32_t* overflow;
    float* io;        // dense output (decode_dense only)
    int tp;           // TMA kernel: positions per tile
    int n_tiles;      // TMA kernel: total tiles
    int use_tmap;     // TMA kernel: 1 = one 2-D tensor-map copy per tile, 0 = one 1-D bulk copy per channel row
    alignas(64) CUtensorMap tmap[YOLO_B200_MAX_SCALES];   // [positions x (batch*na*(5+nc)) rows] per aligned scale
};

#ifndef YB_DC_THREADS
#define YB_DC_THREADS 128
#endif
#ifndef YB_DC_UNROLL
#define YB_DC_UNROLL 16
#endif
#ifndef YB_DC_UNROLL1
#define YB_DC_UNROLL1 40   // batch size of the scalar-load path (planes not a multiple of 4 floats)
#endif
#ifndef YB_DC_MINBLOCKS
#define YB_DC_MINBLOCKS 4
#endif
#ifndef YB_DC_SMEM_PAD
#define YB_DC_SMEM_PAD 0   // unused dynamic shared memory per CTA: caps the resident CTAs per SM below what the registers allow
#endif

constexpr int kDcThreads = YB_DC_THREADS;   // decode_compact CTA size

// Head element types of the LDG decode_compact kernels: float, __half, __nv_bfloat16.  A 16-bit value is converted to fp32
// right after the load; the conversion is exact, so everything after it is the fp32 code on the values h.float() holds.
template <typename T> __device__ __forceinline__ float f32_of_bits(unsigned short b);
template <> __device__ __forceinline__ float f32_of_bits<__half>(unsigned short b) { return __half2float(__ushort_as_half(b)); }
template <> __device__ __forceinline__ float f32_of_bits<__nv_bfloat16>(unsigned short b) {
    return __bfloat162float(__ushort_as_bfloat16(b));
}
__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }

// VEC consecutive elements at p as fp32: one 16-byte (fp32) or 8-byte (16-bit) streaming load for VEC = 4
template <int VEC, typename T>
__device__ __forceinline__ void load_vec(float (&dst)[VEC], const T* p) {
    if constexpr (std::is_same_v<T, float>) {
        if constexpr (VEC == 4) {
            const float4 v = ldg_stream4(p);
            dst[0] = v.x; dst[1] = v.y; dst[2] = v.z; dst[3] = v.w;
        } else {
            dst[0] = ldg_stream(p);
        }
    } else if constexpr (VEC == 4) {
        const uint2 v = ldg_stream_b16x4(p);                       // element 0 in the low half of v.x
        dst[0] = f32_of_bits<T>((unsigned short)(v.x & 0xffffu)); dst[1] = f32_of_bits<T>((unsigned short)(v.x >> 16));
        dst[2] = f32_of_bits<T>((unsigned short)(v.y & 0xffffu)); dst[3] = f32_of_bits<T>((unsigned short)(v.y >> 16));
    } else {
        dst[0] = f32_of_bits<T>(ldg_stream_b16(p));
    }
}

// Exact class pick in sigmoid space: first k maximising sigma(logit_k) (torch.max semantics on the
// decoded tensor, reference utils.py:212).  Only reached when the two largest logits collapse to
// (nearly) the same fp32 sigmoid, e.g. logits {20, 25} -> both 1.0 (SURVEY.md section 7 hard parts).
template <typename T>
__device__ __noinline__ void rescan_classes(const T* cls0, int stride, int nc, float& conf, int& cls) {
    float best = -1.0f;
    int bi = 0;
    for (int k = 0; k < nc; ++k) {
        const float s = sigmoidf_rn(to_f32(cls0[(size_t)k * stride]));       // generic load: global planes or a shared-memory tile
        if (s > best) { best = s; bi = k; }
    }
    conf = best;
    cls = bi;
}

// Everything after the class scan, for ONE anchor: scores, thresholds, box decode, warp-aggregated emission.
// Shared by the LDG and the TMA kernel so that both produce bit-identical candidates.  All 32 lanes call.
//   t0..t4   raw x, y, w, h, objectness logits          m / m2 / idx  max, second max, first arg-max class logit
//   cls0     address of this anchor's class-0 logit, consecutive classes `cls_stride` elements apart
template <typename T>
__device__ __forceinline__ void finish_anchor(const DecodeParams& P, const ScaleDev& S, bool active, int img, int a, int pos,
                                              float t0, float t1, float t2, float t3, float t4,
                                              float m, float m2, int idx, const T* cls0, int cls_stride) {
    const int nc = P.nc;
    const float stride = S.stride;
    const float conf = P.conf;
    // more than twice the worst-case relative error eps of one sigmoid evaluation (eps <= 4.2e-7 + 7.3e-8 * |x|, < 6.9e-6
    // for |x| <= 88, see common.cuh): if sigma(second largest logit) is further than this below sigma(largest), no other
    // class can reach the max.  That needs kSlack * (1 - 2^-24) >= (1 + eps) / (1 - eps): 1.00003 against 1.0000138
    const float kSlack = 1.00003f;
    bool emit = false;
    yolo_b200_box box = {0.f, 0.f, 0.f, 0.f};
    float score = 0.f, cls_conf = 1.0f;
    int cls = 0;
    if (active) {
        const float so = sigmoidf_rn(t4);
        const float sm = (nc > 1) ? sigmoidf_rn(m) : 1.0f;     // n_classes == 1: column 5 := 1 (yolo_layer.py:95-96)
        // cheap reject; NaN anywhere in obj / class logits makes the comparison false
        if (so * sm * kSlack > conf) {
            cls_conf = sm;
            cls = idx;
            if (nc > 1 && sigmoidf_rn(m2) * kSlack >= sm) rescan_classes(cls0, cls_stride, nc, cls_conf, cls);
            score = __fmul_rn(so, cls_conf);                     // utils.py:213
            if (score > conf) {                                   // utils.py:216
                const float w = decode_wh(t2, S.av[a][0], stride);
                const float h = decode_wh(t3, S.av[a][1], stride);
                if (w > P.min_wh && h > P.min_wh && finitef(w) && finitef(h)) {   // utils.py:217-218
                    const int gy = pos / S.nx;
                    const int gx = pos - gy * S.nx;
                    const float x = decode_xy(t0, (float)gx, stride);
                    const float y = decode_xy(t1, (float)gy, stride);
                    if (finitef(x) && finitef(y)) {
                        emit = true;
                        box = to_corners(x, y, w, h);            // utils.py:231
                    }
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

// One work unit of the LDG kernels: VEC consecutive positions of one (image, anchor) slab.  Units past the end are
// clamped onto the last one (a valid address) and marked inactive, so that the lane still takes part in the collectives.
template <typename T>
struct DcUnit {
    const T* base;       // channel 0 of the unit's first position
    int img, a, pos0;
    bool active;
};

template <int VEC, typename T>
__device__ __forceinline__ DcUnit<T> dc_unit(const ScaleDev& S, int no, int unit) {
    DcUnit<T> u;
    u.active = unit < S.n_units;
    if (!u.active) unit = S.n_units - 1;
    const int pv_per_slab = S.plane / VEC;
    const int slab = unit / pv_per_slab;
    const int pv = unit - slab * pv_per_slab;
    u.img = slab / S.na;
    u.a = slab - u.img * S.na;
    u.pos0 = pv * VEC;
    u.base = static_cast<const T*>(S.head) + (size_t)slab * no * S.plane + u.pos0;
    return u;
}

// Running (max, second max, first arg-max) over the class planes at cbase, kDcUnroll planes in flight per batch; the max
// propagates NaN.
template <int VEC, int kDcUnroll, typename T>
__device__ __forceinline__ void scan_classes(const T* cbase, int plane, int nc, float (&m)[VEC], float (&m2)[VEC],
                                             int (&idx)[VEC]) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) { m[j] = __int_as_float(0xff800000); m2[j] = m[j]; idx[j] = 0; }
    int c0 = 0;
    auto scan = [&](const float (&v)[kDcUnroll][VEC], int cfirst) {
#pragma unroll
        for (int u = 0; u < kDcUnroll; ++u) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const float x = v[u][j];
                const bool up = x > m[j];
                m2[j] = up ? m[j] : fmaxf(m2[j], x);
                idx[j] = up ? (cfirst + u) : idx[j];
                m[j] = fmax_nan(m[j], x);
            }
        }
    };
    auto fetch = [&](float (&v)[kDcUnroll][VEC], int cfirst) {
#pragma unroll
        for (int u = 0; u < kDcUnroll; ++u) load_vec<VEC>(v[u], cbase + (size_t)(cfirst + u) * plane);
    };
    if (nc > 1) {
        for (; c0 + kDcUnroll <= nc; c0 += kDcUnroll) {
            float v[kDcUnroll][VEC];
            fetch(v, c0);
            scan(v, c0);
        }
        for (; c0 < nc; ++c0) {
            float v[VEC];
            load_vec<VEC>(v, cbase + (size_t)c0 * plane);
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const float x = v[j];
                const bool up = x > m[j];
                m2[j] = up ? m[j] : fmaxf(m2[j], x);
                idx[j] = up ? c0 : idx[j];
                m[j] = fmax_nan(m[j], x);
            }
        }
    }
}

// Dense: one unit per thread, every plane read.
template <int VEC, int kDcUnroll, typename T>
__device__ __forceinline__ void decode_compact_dense_body(const DecodeParams& P, const ScaleDev& S, int block_local) {
    const int plane = S.plane;
    const DcUnit<T> u = dc_unit<VEC, T>(S, P.nc + 5, block_local * kDcThreads + (int)threadIdx.x);

    // box + objectness planes
    float t[5][VEC];
#pragma unroll
    for (int c = 0; c < 5; ++c) load_vec<VEC>(t[c], u.base + (size_t)c * plane);

    float m[VEC], m2[VEC];
    int idx[VEC];
    const T* cbase = u.base + (size_t)5 * plane;
    scan_classes<VEC, kDcUnroll, T>(cbase, plane, P.nc, m, m2, idx);

#pragma unroll
    for (int j = 0; j < VEC; ++j)
        finish_anchor(P, S, u.active, u.img, u.a, u.pos0 + j, t[0][j], t[1][j], t[2][j], t[3][j], t[4][j],
                      m[j], m2[j], idx[j], cbase + j, plane);
}

// Objectness gate.  finish_anchor's first test is fl(fl(so * sm) * kSlack) > conf with so = sigmoidf_rn(t4) and
// sm = sigmoidf_rn(max class logit) (or 1 for one class).  sigmoidf_rn ends in rcp.approx(1 + e) with 1 + e >= 1, and
// rcp.approx is within 1 ulp, so sm <= 1 + 2^-23; with the two roundings the left side is at most
// so * 1.00003 * (1 + 2^-23) * (1 + 2^-24)^2 < so * 1.0000305 for so >= 0.  The gate computes fl(so * 1.0001), which is
// >= so * 1.0001 * (1 - 2^-24) > so * 1.0000305: whenever the test can pass, the gate passes.  so is the very value
// finish_anchor computes from the same t4.  NaN objectness gives so = NaN and a false gate, as the test is false there
// too; -inf gives so = 0, which passes only if conf < 0, like the test.
__device__ __forceinline__ bool obj_gate(float t4, float conf) {
    return __fmul_rn(sigmoidf_rn(t4), 1.0001f) > conf;
}

// Gated: one unit per thread, as in the dense kernel, but the objectness plane is read first and the box and class
// planes only for units with a position that passes obj_gate, so only the 32-byte sectors some passing anchor needs are
// requested.  With every position passing, a thread issues the loads of the dense kernel, one round trip later.
// (Variants that prefetch the objectness of a second or fourth unit per thread while scanning the current one were
// slower on every configuration but conf 0.001: DESIGN.md section 6.)
template <int VEC, int kDcUnroll, typename T>
__device__ __forceinline__ void decode_compact_gated_body(const DecodeParams& P, const ScaleDev& S, int block_local) {
    const int plane = S.plane;
    const DcUnit<T> u = dc_unit<VEC, T>(S, P.nc + 5, block_local * kDcThreads + (int)threadIdx.x);
    float t[5][VEC];
    load_vec<VEC>(t[4], u.base + (size_t)4 * plane);
    bool gate[VEC];
    bool any = false;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
        gate[j] = u.active && obj_gate(t[4][j], P.conf);
        any |= gate[j];
    }
    float m[VEC], m2[VEC];
    int idx[VEC];
    const T* cbase = u.base + (size_t)5 * plane;
    if (any) {
#pragma unroll
        for (int c = 0; c < 4; ++c) load_vec<VEC>(t[c], u.base + (size_t)c * plane);
        scan_classes<VEC, kDcUnroll, T>(cbase, plane, P.nc, m, m2, idx);
    } else {                                                   // finish_anchor reads none of these for a gated-off position
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            t[0][j] = t[1][j] = t[2][j] = t[3][j] = 0.0f;
            m[j] = m2[j] = 0.0f;
            idx[j] = 0;
        }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j)
        finish_anchor(P, S, gate[j], u.img, u.a, u.pos0 + j, t[0][j], t[1][j], t[2][j], t[3][j], t[4][j],
                      m[j], m2[j], idx[j], cbase + j, plane);
}

__device__ __forceinline__ const ScaleDev& dc_scale(const DecodeParams& P) {
    int s = 0;
#pragma unroll
    for (int k = 1; k < YOLO_B200_MAX_SCALES; ++k)
        if (k < P.n_scales && (int)blockIdx.x >= P.sc[k].first_block) s = k;
    return P.sc[s];
}

// T: the element type of every head of the launch (float, __half, __nv_bfloat16)
template <typename T>
__global__ void __launch_bounds__(kDcThreads, YB_DC_MINBLOCKS)
decode_compact_kernel(const __grid_constant__ DecodeParams P) {
    const ScaleDev& S = dc_scale(P);
    const int block_local = (int)blockIdx.x - S.first_block;
    if (S.vec == 4) decode_compact_gated_body<4, YB_DC_UNROLL, T>(P, S, block_local);
    else            decode_compact_gated_body<1, YB_DC_UNROLL1, T>(P, S, block_local);
}

template <typename T>
__global__ void __launch_bounds__(kDcThreads, YB_DC_MINBLOCKS)
decode_compact_dense_kernel(const __grid_constant__ DecodeParams P) {
    const ScaleDev& S = dc_scale(P);
    const int block_local = (int)blockIdx.x - S.first_block;
    if (S.vec == 4) decode_compact_dense_body<4, YB_DC_UNROLL, T>(P, S, block_local);
    else            decode_compact_dense_body<1, YB_DC_UNROLL1, T>(P, S, block_local);
}

// ---- mbarrier / TMA bulk-copy helpers --------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t phase) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(phase) : "memory");
}
// 1-D TMA bulk copy global -> shared, completion signalled on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}


// 2-D tiled TMA load (SASS: UTMALDG): box = [tp positions] x [5+nc channel rows] of one (image, anchor) slab
__device__ __forceinline__ void tma_tile_g2s(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(x), "r"(y), "r"(smem_u32(bar)) : "memory");
}

// ------------------------------------------------------------------------------------------------
// TMA variant of the fused kernel: persistent CTAs (one per SM), a 2-stage shared-memory ring filled by
// 1-D bulk copies (cp.async.bulk + mbarrier complete_tx; SASS UBLKCP), one producer warp and 8 consumer
// warps.  A tile = up to `tp` consecutive positions of one (image, anchor) slab x all 5+nc channel planes,
// i.e. 5+nc bulk copies of tp*4 bytes.  While the consumers scan stage s, the copies of the next tile are in
// flight, so HBM requests never drain.  Planes whose size is not a multiple of 4 floats (19x19, 13x13) are not
// 16-byte aligned per channel: those tiles are filled by the consumers with plain coalesced loads.
constexpr int kTcConsumers = 256;
constexpr int kTcThreads = kTcConsumers + 32;
constexpr int kTcStages = 2;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void consumer_bar_sync() {            // named barrier 1: the 256 consumer threads only
    asm volatile("bar.sync 1, %0;" ::"n"(kTcConsumers) : "memory");
}

__global__ void __launch_bounds__(kTcThreads, 1)
decode_compact_tma_kernel(const __grid_constant__ DecodeParams P) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t full[kTcStages];
    __shared__ __align__(8) uint64_t empty[kTcStages];
    const int tid = threadIdx.x;
    const int nc = P.nc, no = nc + 5, tp = P.tp;
    const int stage_floats = no * tp;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kTcStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kTcConsumers / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto locate = [&](int tile, int& sc, int& slab, int& p0) {
        sc = 0;
#pragma unroll
        for (int k = 1; k < YOLO_B200_MAX_SCALES; ++k)
            if (k < P.n_scales && tile >= P.sc[k].first_tile) sc = k;
        const int local = tile - P.sc[sc].first_tile;
        slab = local / P.sc[sc].tiles_per_slab;
        p0 = (local - slab * P.sc[sc].tiles_per_slab) * tp;
    };

    if (tid >= kTcConsumers) {
        // ===== producer warp =====
        const int lane = tid & 31;
        int it = 0;
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            const int st = it % kTcStages;
            mbar_wait(&empty[st], ((it / kTcStages) & 1) ^ 1);         // consumers released this stage
            int sc, slab, p0;
            locate(tile, sc, slab, p0);
            const ScaleDev& S = P.sc[sc];
            if (S.vec != 4) continue;                                  // unaligned plane: the consumers fill the stage
            float* dst = smem + (size_t)st * stage_floats;
            if (P.use_tmap) {
                // one tensor-map copy brings the whole [5+nc] x [tp] tile; positions past the plane end are zero-filled
                if (lane == 0) {
                    mbar_expect_tx(&full[st], (uint32_t)stage_floats * 4u);
                    tma_tile_g2s(dst, &P.tmap[sc], p0, slab * no, &full[st]);
                }
                continue;
            }
            const int np = min(tp, S.plane - p0);
            const uint32_t bytes = (uint32_t)np * 4u;
            if (lane == 0) mbar_expect_tx(&full[st], bytes * (uint32_t)no);
            __syncwarp();
            const float* src = static_cast<const float*>(S.head) + (size_t)slab * no * S.plane + p0;
            for (int c = lane; c < no; c += 32)
                tma_bulk_g2s(dst + (size_t)c * tp, src + (size_t)c * S.plane, bytes, &full[st]);
        }
        return;
    }

    // ===== consumer warps: one position per thread =====
    // full[] completes a phase only for TMA-filled tiles, so its parity is tracked per stage (empty[] completes
    // once per use of the stage, whoever filled it).
    uint32_t full_parity = 0;
    int it = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
        const int st = it % kTcStages;
        int sc, slab, p0;
        locate(tile, sc, slab, p0);
        const ScaleDev& S = P.sc[sc];
        const int np = min(tp, S.plane - p0);
        float* tl = smem + (size_t)st * stage_floats;
        if (S.vec == 4) {
            mbar_wait(&full[st], (full_parity >> st) & 1u);
            full_parity ^= 1u << st;
        } else {
            consumer_bar_sync();                                       // nobody still reads this stage
            const float* src = static_cast<const float*>(S.head) + (size_t)slab * no * S.plane + p0;
            // a warp copies one channel row at a time, 8 loads in flight per lane
            for (int c = tid >> 5; c < no; c += kTcConsumers / 32) {
                const float* row = src + (size_t)c * S.plane;
                float v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) { const int p = (tid & 31) + 32 * k; v[k] = p < np ? ldg_stream(row + p) : 0.0f; }
#pragma unroll
                for (int k = 0; k < 8; ++k) { const int p = (tid & 31) + 32 * k; if (p < np) tl[c * tp + p] = v[k]; }
            }
            consumer_bar_sync();
        }
        const bool active = tid < np;
        const int p = active ? tid : 0;
        const float* col = tl + p;
        const float t0 = col[0], t1 = col[tp], t2 = col[2 * tp], t3 = col[3 * tp], t4 = col[4 * tp];
        float m = __int_as_float(0xff800000), m2 = m;
        int idx = 0;
        const float* cls0 = col + 5 * tp;
        if (nc > 1) {
#pragma unroll 8
            for (int c = 0; c < nc; ++c) {
                const float x = cls0[c * tp];
                const bool up = x > m;
                m2 = up ? m : fmaxf(m2, x);
                idx = up ? c : idx;
                m = fmax_nan(m, x);
            }
        }
        const int img = slab / S.na;
        const int a = slab - img * S.na;
        finish_anchor(P, S, active, img, a, p0 + p, t0, t1, t2, t3, t4, m, m2, idx, cls0, tp);
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&empty[st]);
    }
}

// ------------------------------------------------------------------------------------------------
// Dense decode: (B, na*no, ny, nx) channel-major planes -> (B, N, no) row-major rows.
// One CTA = kDdPos positions of one (image, anchor) slab x all `no` channels, transposed through
// shared memory: global reads are 128-byte coalesced per channel, global writes are one contiguous
// run of np*no floats (16-byte vector stores; the tile is shifted inside shared memory so that
// shared and global addresses have the same 16-byte phase).
constexpr int kDdPos = 128;
constexpr int kDdThreads = 256;
constexpr int kDdUnroll = 5;     // loads in flight per thread and batch (128-bit path: 5 x 8 warps = 40 channels)

__device__ __forceinline__ int dd_tiles_per_slab(int plane) { return (plane + kDdPos - 1) / kDdPos; }

__global__ void __launch_bounds__(kDdThreads)
decode_dense_kernel(const __grid_constant__ DecodeParams P) {
    extern __shared__ __align__(128) float smem[];
    int s = 0;
#pragma unroll
    for (int k = 1; k < YOLO_B200_MAX_SCALES; ++k)
        if (k < P.n_scales && (int)blockIdx.x >= P.sc[k].first_block) s = k;
    const ScaleDev& S = P.sc[s];
    const int nc = P.nc, no = nc + 5, plane = S.plane;
    const int tps = dd_tiles_per_slab(plane);
    const int block_local = (int)blockIdx.x - S.first_block;
    const int slab = block_local / tps;
    const int tile = block_local - slab * tps;
    const int img = slab / S.na;
    const int a = slab - img * S.na;
    const int p0 = tile * kDdPos;
    const int np = min(kDdPos, plane - p0);

    const size_t out_off = ((size_t)img * P.rows_per_img + S.row_off + (size_t)a * plane + p0) * no;
    const int mis = (int)(out_off & 3);
    float* tl = smem + mis;

    if (S.vec == 4) {
        // 128-bit path (plane a multiple of 4 floats): one warp covers the tile's 128 positions of one channel with
        // a single LDG.128 per lane; the 8 warps take channels round-robin.  The number of outstanding requests per
        // SM is limited, so 512-byte requests are what keeps enough bytes in flight (profiles/r01_e_dense_decode.txt).
        // Shared-memory stores: lane l holds positions 4l..4l+3; in store k it writes position 4l + ((k + l/8) & 3),
        // which makes the 32 addresses of one store hit 32 different banks (row pitch 5+nc is odd).
        const int warp = (int)threadIdx.x >> 5, lane = (int)threadIdx.x & 31, g = lane >> 3;
        if (4 * lane < np) {
            const float* src = static_cast<const float*>(S.head) + (size_t)slab * no * plane + p0 + 4 * lane;
            const float stride = S.stride;
            float* drow[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) drow[k] = tl + (4 * lane + ((k + g) & 3)) * no;
            auto put = [&](int ch, const float (&r)[4]) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float val = g == 0 ? r[k] : g == 1 ? r[(k + 1) & 3] : g == 2 ? r[(k + 2) & 3] : r[(k + 3) & 3];
                    drow[k][ch] = val;
                }
            };
            int c = warp;
            if (c < 4) {                                   // the box channels: warps 0..3, first round
                const float4 t = ldg_stream4(src + (size_t)c * plane);
                const float tv[4] = {t.x, t.y, t.z, t.w};
                float r[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int pos = p0 + 4 * lane + j;
                    const int gy = pos / S.nx, gx = pos - gy * S.nx;
                    r[j] = c == 0 ? decode_xy(tv[j], (float)gx, stride)
                         : c == 1 ? decode_xy(tv[j], (float)gy, stride)
                                  : decode_wh(tv[j], S.av[a][c - 2], stride);
                }
                put(c, r);
                c += kDdThreads / 32;
            }
            const float* q = src + (size_t)c * plane;
            const size_t qstep = (size_t)(kDdThreads / 32) * plane;
            for (; c + (kDdUnroll - 1) * (kDdThreads / 32) < no; c += kDdUnroll * (kDdThreads / 32)) {
                float4 v[kDdUnroll];
#pragma unroll
                for (int u = 0; u < kDdUnroll; ++u, q += qstep) v[u] = ldg_stream4(q);
#pragma unroll
                for (int u = 0; u < kDdUnroll; ++u) {
                    const float r[4] = {sigmoidf_rn(v[u].x), sigmoidf_rn(v[u].y), sigmoidf_rn(v[u].z), sigmoidf_rn(v[u].w)};
                    put(c + u * (kDdThreads / 32), r);
                }
            }
            for (; c < no; c += kDdThreads / 32, q += qstep) {
                const float4 t = ldg_stream4(q);
                const float r[4] = {sigmoidf_rn(t.x), sigmoidf_rn(t.y), sigmoidf_rn(t.z), sigmoidf_rn(t.w)};
                put(c, r);
            }
            if (nc == 1 && warp == 5) {                    // single-class models: column 5 := 1 (yolo_layer.py:95-96)
                const float one[4] = {1.0f, 1.0f, 1.0f, 1.0f};
                put(5, one);
            }
        }
    } else {
        const int p = (int)threadIdx.x % kDdPos;
        const int half = (int)threadIdx.x / kDdPos;
        // channel split between the two halves of the CTA: half 0 takes the four box channels (two of them need the
        // slower expf) plus the first n0 sigmoid channels, half 1 the remaining sigmoid channels
        const int n_sig = no - 4;
        const int n0 = n_sig > 4 ? (n_sig - 4) / 2 : 0;
        if (p < np) {
            const float* src = static_cast<const float*>(S.head) + (size_t)slab * no * plane + p0 + p;
            float* dst = tl + p * no;
            const float stride = S.stride;
            if (half == 0) {
                const int pos = p0 + p;
                const int gy = pos / S.nx, gx = pos - gy * S.nx;
                const float t0 = ldg_stream(src), t1 = ldg_stream(src + plane);
                const float t2 = ldg_stream(src + 2 * (size_t)plane), t3 = ldg_stream(src + 3 * (size_t)plane);
                dst[0] = decode_xy(t0, (float)gx, stride);
                dst[1] = decode_xy(t1, (float)gy, stride);
                dst[2] = decode_wh(t2, S.av[a][0], stride);
                dst[3] = decode_wh(t3, S.av[a][1], stride);
            }
            int c = half ? 4 + n0 : 4;
            const int c_end = half ? no : 4 + n0;
            const float* q = src + (size_t)c * plane;          // walks down the channel planes
            float* d = dst + c;
            for (; c + kDdUnroll <= c_end; c += kDdUnroll, d += kDdUnroll) {
                float v[kDdUnroll];
    #pragma unroll
                for (int u = 0; u < kDdUnroll; ++u, q += plane) v[u] = ldg_stream(q);
    #pragma unroll
                for (int u = 0; u < kDdUnroll; ++u) d[u] = sigmoidf_rn(v[u]);
            }
            for (; c < c_end; ++c, ++d, q += plane) *d = sigmoidf_rn(ldg_stream(q));
            if (nc == 1 && half == 1) dst[5] = 1.0f;            // single-class models: column 5 := 1 (yolo_layer.py:95-96)
        }
    }
    __syncthreads();

    // contiguous copy-out of np*no floats
    const int n_el = np * no;
    float* out = P.io + out_off;
    const int head = min(n_el, (4 - mis) & 3);
    if ((int)threadIdx.x < head) out[threadIdx.x] = tl[threadIdx.x];
    const int n4 = (n_el - head) >> 2;
    const float4* s4 = reinterpret_cast<const float4*>(tl + head);
    float4* o4 = reinterpret_cast<float4*>(out + head);
    for (int i = threadIdx.x; i < n4; i += kDdThreads) o4[i] = s4[i];
    const int done = head + (n4 << 2);
    if ((int)threadIdx.x < n_el - done) out[done + threadIdx.x] = tl[done + threadIdx.x];
}

// ------------------------------------------------------------------------------------------------
// TMA variant of the dense decode: persistent CTAs (one per SM), 8 consumer warps + 1 producer warp.
//   in   a ring of [5+nc] x [128 positions] tiles filled by one 2-D tensor-map copy each (UTMALDG).  Scales whose planes
//        are not a multiple of 4 floats (19x19, 13x13) cannot be described by a tensor map (16-byte row pitch): the host
//        gives those to the LDG kernel in a second launch and this kernel's tile table skips them
//   out  the transposed [positions] x [5+nc] tile is built in a second set of shared-memory buffers and leaves as ONE
//        bulk copy shared -> global (cp.async.bulk, UBLKCP) of the 16-byte aligned body of the np*(5+nc) contiguous
//        floats; the <= 3 floats before and after it are stored by three threads
// Loads of the next tiles and the store of the previous tile are in flight while the consumers transform the current
// one, so neither direction of the HBM stream drains (the LDG kernel alternates a load phase and a store phase per CTA).
struct DenseTmaParams {
    int stages_in, bufs_out;
};

__device__ __forceinline__ void bulk_s2g(void* gdst, const void* ssrc, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(ssrc)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

constexpr int kDtMaxStages = 4;

__global__ void __launch_bounds__(kTcThreads, 1)
decode_dense_tma_kernel(const __grid_constant__ DecodeParams P, const DenseTmaParams Q) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t full[kDtMaxStages];
    __shared__ __align__(8) uint64_t empty[kDtMaxStages];
    const int tid = threadIdx.x;
    const int nc = P.nc, no = nc + 5;
    constexpr int tp = kDdPos;
    const int stage_floats = no * tp;
    const int out_floats = stage_floats + 4;                     // + phase slack
    float* out_base = smem + (size_t)Q.stages_in * stage_floats;

    if (tid == 0) {
        for (int s = 0; s < Q.stages_in; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], kTcConsumers / 32); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto locate = [&](int tile, int& sc, int& slab, int& p0) {
        sc = 0;
#pragma unroll
        for (int k = 1; k < YOLO_B200_MAX_SCALES; ++k)
            if (k < P.n_scales && tile >= P.sc[k].first_tile) sc = k;
        const int local = tile - P.sc[sc].first_tile;
        slab = local / P.sc[sc].tiles_per_slab;
        p0 = (local - slab * P.sc[sc].tiles_per_slab) * tp;
    };

    if (tid >= kTcConsumers) {
        // ===== producer: one elected thread =====
        if ((tid & 31) != 0) return;
        int it = 0, st = 0;
        uint32_t ph = 1;                                          // first pass over the ring: the stages are free
        for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
            mbar_wait(&empty[st], ph);
            int sc, slab, p0;
            locate(tile, sc, slab, p0);
            mbar_expect_tx(&full[st], (uint32_t)stage_floats * 4u);
            tma_tile_g2s(smem + (size_t)st * stage_floats, &P.tmap[sc], p0, slab * no, &full[st]);
            if (++st == Q.stages_in) { st = 0; ph ^= 1u; }
        }
        return;
    }

    // ===== consumers =====
    const int p = tid & (tp - 1), half = tid >> 7;
    const int n_sig = no - 4;
    const int n0 = n_sig > 4 ? (n_sig - 4) / 2 : 0;               // half 0: box channels (two expf) + n0 sigmoid channels
    uint32_t full_parity = 0;
    int it = 0, st = 0, ob = 0;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
        int sc, slab, p0;
        locate(tile, sc, slab, p0);
        const ScaleDev& S = P.sc[sc];
        const int np = min(tp, S.plane - p0);
        const int img = slab / S.na;
        const int a = slab - img * S.na;
        float* in = smem + (size_t)st * stage_floats;
        // the bulk store that last read output buffer `ob` must have finished reading it
        if (tid == 0) { if (Q.bufs_out == 2) bulk_wait_read<1>(); else bulk_wait_read<0>(); }
        consumer_bar_sync();
        mbar_wait(&full[st], (full_parity >> st) & 1u);
        full_parity ^= 1u << st;

        const size_t out_off = ((size_t)img * P.rows_per_img + S.row_off + (size_t)a * S.plane + p0) * no;
        const int mis = (int)(out_off & 3);
        float* tl = out_base + (size_t)ob * out_floats + mis;
        if (p < np) {
            const float* col = in + p;
            float* dst = tl + p * no;
            const float stride = S.stride;
            if (half == 0) {
                const int pos = p0 + p;
                const int gy = pos / S.nx, gx = pos - gy * S.nx;
                dst[0] = decode_xy(col[0], (float)gx, stride);
                dst[1] = decode_xy(col[tp], (float)gy, stride);
                dst[2] = decode_wh(col[2 * tp], S.av[a][0], stride);
                dst[3] = decode_wh(col[3 * tp], S.av[a][1], stride);
            }
            int c = half ? 4 + n0 : 4;
            const int c_end = half ? no : 4 + n0;
            for (; c + 8 <= c_end; c += 8) {
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = col[(c + u) * tp];
#pragma unroll
                for (int u = 0; u < 8; ++u) dst[c + u] = sigmoidf_rn(v[u]);
            }
            for (; c < c_end; ++c) dst[c] = sigmoidf_rn(col[c * tp]);
            if (nc == 1 && half == 1) dst[5] = 1.0f;              // single-class models: column 5 := 1 (yolo_layer.py:95-96)
        }
        fence_proxy_async_smem();                                 // generic-proxy writes -> visible to the bulk copy
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&empty[st]);             // the input stage is free again
        consumer_bar_sync();

        const int n_el = np * no;
        float* out = P.io + out_off;
        const int head = min(n_el, (4 - mis) & 3);
        const int n4 = (n_el - head) >> 2;
        const int done = head + (n4 << 2);
        if (tid == 0) {                                           // (an empty group keeps the group count = tile count)
            if (n4 > 0) bulk_s2g(out + head, tl + head, (uint32_t)n4 * 16u);
            bulk_commit();
        }
        if (tid >= 32 && tid < 32 + head) out[tid - 32] = tl[tid - 32];
        if (tid >= 64 && tid < 64 + (n_el - done)) out[done + tid - 64] = tl[done + tid - 64];

        if (++st == Q.stages_in) st = 0;
        if (++ob == Q.bufs_out) ob = 0;
    }
    if (tid == 0) bulk_wait_read<0>();                            // shared memory must outlive the last bulk store
}

// ------------------------------------------------------------------------------------------------
// compact_from_dense: rows of (5+nc) floats, row-major.  Persistent CTAs pull 128-row tiles into a
// 2-stage shared-memory ring with TMA bulk copies (cp.async.bulk + mbarrier complete_tx); one
// thread owns one row and scans it with stride-`no` shared loads (conflict-free for odd `no`).
constexpr int kCfRows = 128;
constexpr int kCfThreads = 128;
constexpr int kCfStages = 2;

struct CompactParams {
    float* pred;
    int batch, rows_per_img, nc;
    long long total_rows;
    int n_tiles;
    int rows_tile;            // rows per tile: <= kCfRows (one thread per row), a multiple of 4 (bulk-copy size rule)
    int use_tma;
    float conf, min_wh;
    int write_back;
    yolo_b200_box* cand_box;
    yolo_b200_meta* cand_meta;
    int cap;
    int32_t* count;
    int32_t* overflow;
};

__global__ void __launch_bounds__(kCfThreads)
compact_from_dense_kernel(const __grid_constant__ CompactParams P) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t full[kCfStages];
    const int no = P.nc + 5;
    const int rows_tile = P.rows_tile;
    const int tile_floats = rows_tile * no;
    const int tid = threadIdx.x;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < kCfStages; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    auto tile_rows = [&](int t) -> int {
        const long long r0 = (long long)t * rows_tile;
        return (int)min((long long)rows_tile, P.total_rows - r0);
    };
    // a tile goes through TMA when it is full (its byte count is a multiple of 16) and the base is aligned
    auto tile_is_tma = [&](int t) -> bool { return P.use_tma && tile_rows(t) == rows_tile; };
    auto issue = [&](int t, int stage) {
        if (tile_is_tma(t)) {
            const uint32_t bytes = (uint32_t)tile_floats * 4u;
            mbar_expect_tx(&full[stage], bytes);
            tma_bulk_g2s(smem + (size_t)stage * tile_floats, P.pred + (size_t)t * tile_floats, bytes, &full[stage]);
        }
    };

    uint32_t phase_bits = 0;
    int t = blockIdx.x;
    if (tid == 0) {
        int tt = t;
#pragma unroll
        for (int s = 0; s < kCfStages; ++s, tt += gridDim.x)
            if (tt < P.n_tiles) issue(tt, s);
    }
    const float inf = __int_as_float(0x7f800000);
    for (int it = 0; t < P.n_tiles; t += gridDim.x, ++it) {
        const int stage = it % kCfStages;
        float* tl = smem + (size_t)stage * tile_floats;
        const int rows = tile_rows(t);
        if (tile_is_tma(t)) {
            mbar_wait(&full[stage], (phase_bits >> stage) & 1u);
            phase_bits ^= 1u << stage;
        } else {
            // tail tile (or unaligned base): plain coalesced copy into the stage
            const float* src = P.pred + (size_t)t * tile_floats;
            for (int i = tid; i < rows * no; i += kCfThreads) tl[i] = src[i];
            __syncthreads();
        }

        bool emit = false;
        yolo_b200_box box = {0.f, 0.f, 0.f, 0.f};
        float score = 0.f, cls_conf = 0.f;
        int cls = 0, img = 0, row = 0;
        if (tid < rows) {
            const long long g = (long long)t * rows_tile + tid;
            img = (int)(g / P.rows_per_img);
            row = (int)(g - (long long)img * P.rows_per_img);
            const float* r = tl + tid * no;
            // first arg-max over the class columns (utils.py:212); fin accumulates 0*v: NaN iff any column is not finite
            float m = r[5], fin = __fmul_rn(r[5], 0.0f);
            int mi = 0;
            for (int k = 1; k < P.nc; ++k) {
                const float v = r[5 + k];
                fin = fmaf(v, 0.0f, fin);
                if (v > m) { m = v; mi = k; }
                m = fmax_nan(m, v);
            }
            const float x = r[0], y = r[1], w = r[2], h = r[3];
            score = __fmul_rn(r[4], m);                                   // utils.py:213
            if (P.write_back) P.pred[(size_t)g * no + 4] = score;
            fin = fmaf(x, 0.0f, fin); fin = fmaf(y, 0.0f, fin); fin = fmaf(w, 0.0f, fin); fin = fmaf(h, 0.0f, fin);
            fin = fmaf(score, 0.0f, fin);
            cls_conf = m;
            cls = mi;
            emit = (score > P.conf) && (w > P.min_wh) && (h > P.min_wh) && (fin == 0.0f) && (fabsf(score) < inf);
            if (emit) box = to_corners(x, y, w, h);
        }
        const int slot = warp_claim_slot(emit, img, P.count);
        if (emit) {
            if (slot < P.cap) store_candidate(P.cand_box, P.cand_meta, (size_t)img * P.cap + slot, box, score, cls_conf, cls, row);
            else atomicMax(P.overflow, 1);
        }
        __syncthreads();                       // everyone is done with this stage
        const int nt = t + kCfStages * gridDim.x;
        if (tid == 0 && nt < P.n_tiles) issue(nt, stage);
    }
}

}  // namespace yb

// ================================================================================================
// host side: argument validation, launch geometry, extern "C" entry points
// ================================================================================================
using namespace yb;

// count[batch] and overflow[1] are zeroed with one memset when the caller laid them out back to back
static cudaError_t zero_counters(int32_t* count, int32_t* overflow, int batch, cudaStream_t stream) {
    if (overflow == count + batch) return cudaMemsetAsync(count, 0, sizeof(int32_t) * (batch + 1), stream);
    cudaError_t e = cudaSuccess;
    if (batch > 0 && (e = cudaMemsetAsync(count, 0, sizeof(int32_t) * batch, stream)) != cudaSuccess) return e;
    return cudaMemsetAsync(overflow, 0, sizeof(int32_t), stream);
}

// esize: bytes per head element (4, or 2 for decode_compact's 16-bit modes)
static int fill_params(DecodeParams& P, const yolo_b200_scale* sc, int n_scales, int batch, int nc,
                       int rows_per_img, bool dense, bool partial = false, int esize = 4) {
    if (!sc) return YOLO_B200_E_NULL;
    if (n_scales < 1 || n_scales > YOLO_B200_MAX_SCALES || batch < 0 || nc < 1 || nc > YOLO_B200_MAX_CLASSES ||
        rows_per_img < 1)
        return YOLO_B200_E_RANGE;
    const int no = nc + 5;
    long long rows = 0, blocks = 0;
    for (int k = 0; k < n_scales; ++k) {
        const yolo_b200_scale& s = sc[k];
        ScaleDev& d = P.sc[k];
        if (!s.head && batch > 0) return YOLO_B200_E_NULL;
        if (s.ny < 1 || s.nx < 1 || s.na < 1 || s.na > YOLO_B200_MAX_ANCHORS || s.row_off < 0) return YOLO_B200_E_RANGE;
        if (((uintptr_t)s.head & (uintptr_t)(esize - 1)) != 0) return YOLO_B200_E_ALIGN;
        d.head = s.head; d.ny = s.ny; d.nx = s.nx; d.na = s.na; d.row_off = s.row_off;
        d.plane = s.ny * s.nx;
        d.stride = s.stride;
        for (int a = 0; a < YOLO_B200_MAX_ANCHORS; ++a) { d.av[a][0] = s.anchor_vec[a][0]; d.av[a][1] = s.anchor_vec[a][1]; }
        // every plane starts at head + (slab*no + c)*plane elements: aligned to 4 elements for all (slab, c) iff
        // plane % 4 == 0 and head is
        d.vec = ((d.plane % 4 == 0) && (((uintptr_t)s.head & (uintptr_t)(4 * esize - 1)) == 0)) ? 4 : 1;
        const long long slabs = (long long)batch * s.na;
        if ((long long)s.row_off + (long long)s.na * d.plane > rows_per_img) return YOLO_B200_E_RANGE;
        if (slabs * d.plane > 0x7fffffffLL) return YOLO_B200_E_RANGE;
        d.n_units = (int)(slabs * d.plane / d.vec);
        rows += (long long)s.na * d.plane;
    }
    // block ranges: scales whose CTAs carry the most work first (128-bit scales, larger planes first), the
    // scalar-load scales last -- their 4x smaller CTAs fill the last, partial wave of the grid.
    // The kernels find their scale by comparing blockIdx.x with first_block, so the table stays sorted by it.
    {
        int order[YOLO_B200_MAX_SCALES];
        for (int k = 0; k < n_scales; ++k) order[k] = k;
        for (int i = 0; i < n_scales; ++i)
            for (int j = i + 1; j < n_scales; ++j) {
                const ScaleDev &a = P.sc[order[i]], &b = P.sc[order[j]];
                const bool swap = dense ? false : (b.vec > a.vec || (b.vec == a.vec && b.plane > a.plane));
                if (swap) { const int t = order[i]; order[i] = order[j]; order[j] = t; }
            }
        ScaleDev sorted[YOLO_B200_MAX_SCALES];
        for (int i = 0; i < n_scales; ++i) {
            ScaleDev& d = sorted[i];
            d = P.sc[order[i]];
            const long long slabs = (long long)batch * d.na;
            d.first_block = (int)blocks;
            if (dense) blocks += slabs * ((d.plane + kDdPos - 1) / kDdPos);
            else       blocks += (d.n_units + kDcThreads - 1) / kDcThreads;
            if (blocks > 0x7fffffffLL) return YOLO_B200_E_RANGE;
        }
        for (int i = 0; i < n_scales; ++i) P.sc[i] = sorted[i];
    }
    for (int k = n_scales; k < YOLO_B200_MAX_SCALES; ++k) { P.sc[k] = P.sc[0]; P.sc[k].first_block = 0x7fffffff; }
    // the scales tile the image's rows exactly, unless the caller decodes only some of them (accumulate mode)
    if (partial ? rows > rows_per_img : rows != rows_per_img) return YOLO_B200_E_RANGE;
    P.n_scales = n_scales; P.batch = batch; P.nc = nc; P.rows_per_img = rows_per_img;
    (void)no;
    return (int)blocks;   // >= 0
}

// Tile geometry of the TMA kernel: the largest tile (positions per channel row) whose 2-stage ring fits in
// shared memory; 0 when even 32 positions do not fit (very large class counts) -> LDG kernel.
static int tma_tile_positions(int no) {
    for (int tp = kTcConsumers; tp >= 32; tp >>= 1)
        if ((size_t)kTcStages * no * tp * sizeof(float) <= 200 * 1024) return tp;
    return 0;
}

// Tile table (first_tile, tiles_per_slab, n_tiles) for tiles of `tp` positions, and -- with_maps -- one 2-D tensor map
// [plane positions] x [batch*na*(5+nc) channel rows], box = [tp] x [5+nc], per scale with 16-byte aligned planes.
static int tile_table(DecodeParams& P, int n_scales, int batch, int no, int tp, bool with_maps, bool aligned_only = false) {
    long long tiles = 0;
    P.tp = tp;
    for (int k = 0; k < n_scales; ++k) {
        P.sc[k].first_tile = (int)tiles;
        P.sc[k].tiles_per_slab = (P.sc[k].plane + tp - 1) / tp;
        // a skipped scale owns no tile: it shares first_tile with its successor, and the kernels' "last scale whose
        // first_tile <= tile" search passes over it
        if (!(aligned_only && P.sc[k].vec != 4)) tiles += (long long)batch * P.sc[k].na * P.sc[k].tiles_per_slab;
    }
    for (int k = n_scales; k < YOLO_B200_MAX_SCALES; ++k) P.sc[k].first_tile = 0x7fffffff;
    if (tiles > 0x7fffffffLL) return YOLO_B200_E_RANGE;
    P.n_tiles = (int)tiles;
    if (!with_maps) return 0;
    if (no > 256) return YOLO_B200_E_RANGE;                             // a TMA box is at most 256 rows
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    const cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess) return (int)e;
    if (!fn || qres != cudaDriverEntryPointSuccess) return YOLO_B200_E_RANGE;
    for (int k = 0; k < n_scales; ++k) {
        if (P.sc[k].vec != 4) continue;                                  // unaligned planes are filled by the consumers
        const cuuint64_t gdim[2] = {(cuuint64_t)P.sc[k].plane, (cuuint64_t)batch * P.sc[k].na * no};
        const cuuint64_t gstride[1] = {(cuuint64_t)P.sc[k].plane * sizeof(float)};
        const cuuint32_t box[2] = {(cuuint32_t)tp, (cuuint32_t)no};
        const cuuint32_t estr[2] = {1, 1};
        const CUresult r = ((EncodeFn)fn)(&P.tmap[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)P.sc[k].head, gdim, gstride,
                                          box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                                          CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return YOLO_B200_E_RANGE;
    }
    return 0;
}

extern "C" int yolo_b200_decode_compact_ex(const yolo_b200_scale* scales, int n_scales, int batch, int nc,
                                           int rows_per_img, float conf_thres, float min_wh,
                                           yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                           int32_t* count, int32_t* overflow, int variant, yolo_b200_stream_t stream) {
    if (!cand_box || !cand_meta || !count || !overflow) return YOLO_B200_E_NULL;
    const bool accumulate = variant >= 0 && (variant & YOLO_B200_VARIANT_ACCUMULATE) != 0;
    if (accumulate) variant &= ~YOLO_B200_VARIANT_ACCUMULATE;
    const int half_bits = variant >= 0 ? variant & (YOLO_B200_VARIANT_F16 | YOLO_B200_VARIANT_BF16) : 0;
    variant &= ~half_bits;
    if (cap_per_img < 1 || variant < 0 || variant > 4) return YOLO_B200_E_RANGE;
    if (half_bits == (YOLO_B200_VARIANT_F16 | YOLO_B200_VARIANT_BF16)) return YOLO_B200_E_RANGE;
    if (half_bits && (variant == 2 || variant == 3)) return YOLO_B200_E_UNSUPPORTED;     // the TMA kernels read fp32 only
    if ((((uintptr_t)cand_box) | ((uintptr_t)cand_meta)) & 15u) return YOLO_B200_E_ALIGN;
    const bool gated = variant <= 1;
    DecodeParams P{};
    const int blocks = fill_params(P, scales, n_scales, batch, nc, rows_per_img, false, accumulate, half_bits ? 2 : 4);
    if (blocks < 0) return blocks;
    P.conf = conf_thres; P.min_wh = min_wh;
    P.cand_box = cand_box; P.cand_meta = cand_meta; P.cap = cap_per_img; P.count = count; P.overflow = overflow;
    cudaError_t e;
    if (!accumulate && (e = zero_counters(count, overflow, batch, stream)) != cudaSuccess) return (int)e;
    if (blocks == 0) return 0;

    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int no = nc + 5;
    const int tp = tma_tile_positions(no);
    // Measured on B200 (profiles/r01_c_decode_variants.txt): the dense LDG kernel streams at 5.8 TB/s, the 1-D bulk-copy
    // ring at 3.1 TB/s (one cp.async.bulk per 1 KB channel row: TMA issue-bound), so "automatic" means LDG, and the gated
    // LDG kernel reads box and class planes only where the objectness can pass (profiles/gated_decode_probe.txt).  The
    // others stay selectable for comparison (2 = 1-D bulk copies, 3 = one 2-D tensor-map copy per tile, 4 = dense LDG).
    const bool use_tma = variant == 2 || variant == 3;
    if (use_tma && tp == 0) return YOLO_B200_E_RANGE;
    P.use_tmap = 0;
    if (use_tma) {
        const int rc = tile_table(P, n_scales, batch, no, tp, variant == 3);
        if (rc != 0) return rc;
        P.use_tmap = variant == 3 ? 1 : 0;
    }
    const long long tiles = P.n_tiles;
    if (use_tma) {
        const size_t smem = (size_t)kTcStages * no * tp * sizeof(float);
        if ((e = cudaFuncSetAttribute(decode_compact_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return (int)e;
        const int grid = (int)(tiles < sms ? tiles : sms);
        decode_compact_tma_kernel<<<grid, kTcThreads, smem, stream>>>(P);
    } else if (half_bits == YOLO_B200_VARIANT_F16) {
        if (gated) decode_compact_kernel<__half><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
        else       decode_compact_dense_kernel<__half><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
    } else if (half_bits == YOLO_B200_VARIANT_BF16) {
        if (gated) decode_compact_kernel<__nv_bfloat16><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
        else       decode_compact_dense_kernel<__nv_bfloat16><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
    } else if (gated) {
        decode_compact_kernel<float><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
    } else {
        decode_compact_dense_kernel<float><<<blocks, kDcThreads, YB_DC_SMEM_PAD, stream>>>(P);
    }
    return (int)cudaGetLastError();
}

extern "C" int yolo_b200_decode_compact(const yolo_b200_scale* scales, int n_scales, int batch, int nc,
                                        int rows_per_img, float conf_thres, float min_wh,
                                        yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                        int32_t* count, int32_t* overflow, yolo_b200_stream_t stream) {
    return yolo_b200_decode_compact_ex(scales, n_scales, batch, nc, rows_per_img, conf_thres, min_wh, cand_box, cand_meta,
                                       cap_per_img, count, overflow, 0, stream);
}

extern "C" int yolo_b200_decode_dense_ex(const yolo_b200_scale* scales, int n_scales, int batch, int nc,
                                         int rows_per_img, float* io, int variant, yolo_b200_stream_t stream) {
    if (!io) return YOLO_B200_E_NULL;
    if ((uintptr_t)io & 15u) return YOLO_B200_E_ALIGN;
    if (variant < 0 || variant > 2) return YOLO_B200_E_RANGE;
    DecodeParams P{};
    const int blocks = fill_params(P, scales, n_scales, batch, nc, rows_per_img, true);
    if (blocks < 0) return blocks;
    P.io = io;
    if (blocks == 0) return 0;
    const int no = nc + 5;
    const size_t tile_bytes = (size_t)kDdPos * no * sizeof(float);
    cudaError_t e;
    // TMA kernel: a ring of input tiles + one or two output tiles in shared memory, as many as fit (85 rows: 3 + 2)
    bool any_aligned = false;
    for (int k = 0; k < n_scales; ++k) any_aligned |= P.sc[k].vec == 4;
    const size_t budget = 226 * 1024;
    DenseTmaParams Q{0, 0};
    if (no <= 256 && any_aligned) {
        if (5 * tile_bytes + 32 <= budget)      Q = {3, 2};
        else if (4 * tile_bytes + 32 <= budget) Q = {2, 2};
        else if (3 * tile_bytes + 16 <= budget) Q = {2, 1};
    }
    if (variant == 2 && Q.stages_in == 0) return YOLO_B200_E_RANGE;
    const size_t ldg_smem = tile_bytes + 4 * sizeof(float);
    if (ldg_smem > 220 * 1024) return YOLO_B200_E_RANGE;   // one 128-position tile of 5+nc rows must fit: nc <= 434
    if ((e = cudaFuncSetAttribute(decode_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ldg_smem)) != cudaSuccess)
        return (int)e;
    if (variant != 1 && Q.stages_in > 0) {
        // aligned scales: TMA kernel; the others: LDG kernel over a block table that skips the aligned scales
        const int rc = tile_table(P, n_scales, batch, no, kDdPos, true, true);
        if (rc != 0) return rc;
        const size_t smem = (size_t)Q.stages_in * tile_bytes + (size_t)Q.bufs_out * (tile_bytes + 16);
        if ((e = cudaFuncSetAttribute(decode_dense_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
            return (int)e;
        int dev = 0, sms = 148;
        if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        const int grid = P.n_tiles < sms ? P.n_tiles : sms;
        decode_dense_tma_kernel<<<grid, kTcThreads, smem, stream>>>(P, Q);
        if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
        long long rest = 0;
        for (int k = 0; k < n_scales; ++k) {
            P.sc[k].first_block = (int)rest;
            if (P.sc[k].vec != 4) rest += (long long)batch * P.sc[k].na * ((P.sc[k].plane + kDdPos - 1) / kDdPos);
        }
        if (rest == 0) return 0;
        decode_dense_kernel<<<(int)rest, kDdThreads, ldg_smem, stream>>>(P);
        return (int)cudaGetLastError();
    }
    decode_dense_kernel<<<blocks, kDdThreads, ldg_smem, stream>>>(P);
    return (int)cudaGetLastError();
}

extern "C" int yolo_b200_decode_dense(const yolo_b200_scale* scales, int n_scales, int batch, int nc,
                                      int rows_per_img, float* io, yolo_b200_stream_t stream) {
    return yolo_b200_decode_dense_ex(scales, n_scales, batch, nc, rows_per_img, io, 0, stream);
}

extern "C" int yolo_b200_compact_from_dense(float* pred, int batch, int rows_per_img, int nc,
                                            float conf_thres, float min_wh, int write_back_score,
                                            yolo_b200_box* cand_box, yolo_b200_meta* cand_meta, int cap_per_img,
                                            int32_t* count, int32_t* overflow, yolo_b200_stream_t stream) {
    if (!cand_box || !cand_meta || !count || !overflow || (!pred && batch > 0)) return YOLO_B200_E_NULL;
    if (batch < 0 || rows_per_img < 1 || nc < 1 || nc > YOLO_B200_MAX_CLASSES || cap_per_img < 1) return YOLO_B200_E_RANGE;
    if (((uintptr_t)pred & 3u) || ((((uintptr_t)cand_box) | ((uintptr_t)cand_meta)) & 15u)) return YOLO_B200_E_ALIGN;
    CompactParams P{};
    P.pred = pred; P.batch = batch; P.rows_per_img = rows_per_img; P.nc = nc;
    P.total_rows = (long long)batch * rows_per_img;
    // rows per tile: as many as fit a 2-stage ring in shared memory (128 for 85-float rows), a multiple of 4
    int rows_tile = kCfRows;
    while (rows_tile > 4 && (size_t)kCfStages * rows_tile * (nc + 5) * sizeof(float) > 200 * 1024) rows_tile >>= 1;
    P.rows_tile = rows_tile;
    const long long tiles = (P.total_rows + rows_tile - 1) / rows_tile;
    if (tiles > 0x7fffffffLL) return YOLO_B200_E_RANGE;
    P.n_tiles = (int)tiles;
    P.use_tma = (((uintptr_t)pred & 15u) == 0) ? 1 : 0;
    P.conf = conf_thres; P.min_wh = min_wh; P.write_back = write_back_score;
    P.cand_box = cand_box; P.cand_meta = cand_meta; P.cap = cap_per_img; P.count = count; P.overflow = overflow;
    cudaError_t e;
    if ((e = zero_counters(count, overflow, batch, stream)) != cudaSuccess) return (int)e;
    if (P.n_tiles == 0) return 0;
    const size_t smem = (size_t)kCfStages * rows_tile * (nc + 5) * sizeof(float);
    if (smem > 200 * 1024) return YOLO_B200_E_RANGE;
    if ((e = cudaFuncSetAttribute(compact_from_dense_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
        return (int)e;
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int per_sm = (int)((220 * 1024) / (smem + 1024));
    const int grid = (int)min((long long)sms * (per_sm < 1 ? 1 : per_sm), tiles);
    compact_from_dense_kernel<<<grid, kCfThreads, smem, stream>>>(P);
    return (int)cudaGetLastError();
}
