// Shared device helpers for the yolo_b200 kernels (sm_100a).
//
// Every arithmetic step that decides a result (decode, score, box corners, IoU) goes through the
// explicit round-to-nearest intrinsics so that nvcc can never contract a*b+c into an FMA: the
// reference computes each torch op with its own fp32 rounding (SURVEY.md App. A / section 7), and the
// fused and dense kernels must produce bit-identical values from the same inputs.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/yolo_b200.h"

namespace yb {

constexpr unsigned kFull = 0xffffffffu;

// ---- streaming global loads (read-once data: do not allocate in L1) -----------------------------
__device__ __forceinline__ float ldg_stream(const float* p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
// 16-bit heads (fp16 / bf16 bit patterns): one element, and four consecutive elements as one 8-byte load
__device__ __forceinline__ unsigned short ldg_stream_b16(const void* p) {
    unsigned short v;
    asm volatile("ld.global.nc.L1::no_allocate.b16 %0, [%1];" : "=h"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ uint2 ldg_stream_b16x4(const void* p) {
    uint2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p));
    return v;
}

// max that propagates NaN (PTX max.NaN.f32, one FMNMX): a NaN anywhere poisons the running max.
__device__ __forceinline__ float fmax_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

// ---- the decode arithmetic (reference models/yolo_layer.py:91-94, SURVEY.md App. A) ---------------
// sigma(x) = 1 / (1 + exp(-x)) on the SFU: one FMUL, MUFU.EX2, one FADD, MUFU.RCP (explicit PTX, so every kernel
// evaluates the identical sequence).  ex2.approx is accurate to 2^-22, fl(1 + e) adds 2^-24 and rcp.approx 1 ulp
// (2^-23): 4.2e-7.  The argument fl(x * fl(-log2 e)) carries the rounding of the product (2^-24) and of log2 e to fp32
// (1.34e-8), which the exponential turns into |x| * 7.3e-8.  So the relative error is <= 4.2e-7 + 7.3e-8 * |x|
// (<= 1.2e-6 for |x| <= 10, < 6.9e-6 up to the fp32 overflow edge |x| = 88) against the 1e-5 the parity criterion
// allows; tests/test_gpu_decode_numerics.py holds every fp32 with 2^-8 <= |x| <= 128 to it, and
// profiles/sigmoid_error_probe.txt has the measured worst case per binade.  An 85-channel row costs
// 170 MUFU operations, which keeps the dense decode kernel HBM-bound instead of issue-bound.  The .ftz forms are
// single instructions; they only differ for results below 1.2e-38 (logits under -87.3), which become 0.
__device__ __forceinline__ float sigmoidf_rn(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__fmul_rn(x, -1.4426950408889634f)));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(__fadd_rn(1.0f, e)));
    return r;
}
// xy: (sigma(t) + grid) * stride   -- add, then multiply, two roundings (yolo_layer.py:91,94)
__device__ __forceinline__ float decode_xy(float t, float grid, float stride) {
    return __fmul_rn(__fadd_rn(sigmoidf_rn(t), grid), stride);
}
// wh: (exp(t) * anchor_vec) * stride                               (yolo_layer.py:92,94)
__device__ __forceinline__ float decode_wh(float t, float anchor, float stride) {
    return __fmul_rn(__fmul_rn(expf(t), anchor), stride);
}
__device__ __forceinline__ bool finitef(float v) { return fabsf(v) < __int_as_float(0x7f800000); }

// xywh -> corners (reference utils/utils.py:56-59): x -+ w/2 (w/2 is exact).
__device__ __forceinline__ yolo_b200_box to_corners(float x, float y, float w, float h) {
    const float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);
    yolo_b200_box b;
    b.x1 = __fsub_rn(x, hw);
    b.y1 = __fsub_rn(y, hh);
    b.x2 = __fadd_rn(x, hw);
    b.y2 = __fadd_rn(y, hh);
    return b;
}

// ---- candidate emission ---------------------------------------------------------------------------
// Reserve `n` consecutive slots of image `img`; returns the first slot (may be >= cap: caller checks).
__device__ __forceinline__ int reserve_slots(int32_t* count, int img, int n) {
    return atomicAdd(count + img, n);
}

__device__ __forceinline__ void store_candidate(yolo_b200_box* cand_box, yolo_b200_meta* cand_meta,
                                                size_t slot, const yolo_b200_box& box, float score,
                                                float cls_conf, int cls, int row) {
    reinterpret_cast<float4*>(cand_box)[slot] = make_float4(box.x1, box.y1, box.x2, box.y2);
    reinterpret_cast<int4*>(cand_meta)[slot] =
        make_int4(__float_as_int(score), __float_as_int(cls_conf), cls, row);
}

// Warp-aggregated compaction for one "does this lane emit" flag.  All 32 lanes must call.
// Lanes of one warp may belong to two different images (tiles straddle image boundaries); the
// aggregation is done per distinct image.  Returns the slot for this lane (or -1).
__device__ __forceinline__ int warp_claim_slot(bool emit, int img, int32_t* count) {
    int slot = -1;
    unsigned pending = __ballot_sync(kFull, emit);
    const int lane = threadIdx.x & 31;
    while (pending) {
        const int leader = __ffs(pending) - 1;
        const int limg = __shfl_sync(kFull, img, leader);
        const unsigned grp = __ballot_sync(kFull, emit && img == limg);
        int base = 0;
        if (lane == leader) base = reserve_slots(count, limg, __popc(grp));
        base = __shfl_sync(kFull, base, leader);
        if (emit && img == limg) slot = base + __popc(grp & ((1u << lane) - 1u));
        pending &= ~grp;
    }
    return slot;
}

}  // namespace yb

// Shared-memory carve-out preference of the kernels that run beside each other in the pipelined detector (decode of batch
// i + 1 next to the NMS kernels of batch i).  Left to the driver, every kernel asks for the split that maximises its own
// occupancy, and on workloads of many small images (tiny-416 batch 1024: 1024-CTA bucket / finalize kernels with 20-odd KB
// of shared memory each) the resulting mix costs 5 % of the step against one common preference of 50 % for all of them;
// with few big images the driver's choice is the best (profiles/r02_y_carveout.txt: cfg 3 168.8 vs 177-181 us, cfg 2 80.3 vs
// 79.2, cfg 4 198.6 vs 191.9).  So: 50 % when an image holds at most kSmallImageRows rows, the default otherwise.
// YOLO_B200_CARVEOUT (percent) overrides both for experiments.
#include <stdlib.h>
constexpr int kSmallImageRows = 4096;
constexpr int kSmallImageCarveout = 50;
inline int yb_carveout_for(long long rows_per_img) {
    static const int env = [] { const char* e = getenv("YOLO_B200_CARVEOUT"); return e && *e ? atoi(e) : -1; }();
    if (env >= 0) return env > 100 ? 100 : env;
    return rows_per_img <= kSmallImageRows ? kSmallImageCarveout : -1;      // -1 = cudaSharedmemCarveoutDefault
}
template <typename K>
inline void yb_prefer_carveout(K kernel, int percent) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, percent);
}
