// Device-side helpers shared by the sm_100a kernels of the observation path (one copy per translation unit:
// everything here lives in an anonymous namespace).
//   agym_ingest.cu    ingest (Atari gray / RGB, DMC), stack
//   agym_observe.cu   fixed fovea (crop / mask / resize_to_full), foveal + peripheral merge
//   agym_flexible.cu  flexible fovea
//   agym_misc.cu      normalise, synthetic frames
//
// Every kernel is a byte/integer streaming kernel bounded by HBM bandwidth or by instruction issue — there is
// no dense contraction on this path, so no tensor cores.  Reference semantics (file:line relative to
// /root/reference/active_gym/) are cited at each kernel; the arithmetic must stay bit-identical to
// oracle/agym_oracle.c for the integer stages (cv2 resize, luma, max, stack, crop, mask, paste) and within
// 0.5 u8 LSB + evaluation error of it for the antialiased resamples.
#pragma once
#include "agym_kernels.cuh"
#ifndef AGYM_EXPERIMENT
#define AGYM_EXPERIMENT 0
#endif

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <utility>
#include <cstdlib>
#include <cstring>

#include "../../include/agym_b200.h"

namespace agym {

namespace {


constexpr int kThreads = 256;

__device__ __forceinline__ uint4 ld_stream128(const void *p) {
    // read-once data (raw simulator frames): bypass L1 allocation
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

struct FastDiv {
    uint32_t magic;
    int32_t d;
    __device__ __forceinline__ explicit FastDiv(int32_t dd) : magic(0xFFFFFFFFu / (uint32_t)dd + 1u), d(dd) {}
    // multiplier from a table of 0xFFFFFFFF / d + 1 (d < 256) instead of an integer division
    __device__ __forceinline__ FastDiv(int32_t dd, const uint32_t *table) : magic(table[dd]), d(dd) {}
    // multiplier computed on the host (0xFFFFFFFF / d + 1)
    __device__ __forceinline__ FastDiv(int32_t dd, uint32_t m) : magic(m), d(dd) {}
    // exact for n * d < 2^32 (all indices here are < 2^24, divisors < 2^8)
    __device__ __forceinline__ int32_t div(int32_t n) const { return d == 1 ? n : (int32_t)__umulhi((uint32_t)n, magic); }
};

__device__ __forceinline__ int clip_rint(double v, double lo, double hi) {
    // np.rint(np.clip(v, lo, hi)): clip first, then round half to even (fov_env.py:166-170)
    return __double2int_rn(fmin(fmax(v, lo), hi));
}

__device__ __forceinline__ uint32_t quant_u8(float v) {
    int q = __float2int_rn(v);
    return (uint32_t)min(max(q, 0), 255);
}

// FOV_RES action of the flexible fovea: fov_res = action (fov_env.py:323).  The reference fails for a window that is
// not an integer size within the frame (float slice bounds; Resize of a window larger than the frame raises); a kernel
// cannot raise, so it truncates, clamps to [1, S] and reports the event in the caller's error word (AGYM_ERR_RES_*).
__device__ __forceinline__ void res_from_action(const DevPlan &p, double a0, double a1, int &rh, int &rw) {
    const bool in_range = a0 >= 1.0 && a0 <= (double)p.S_h && a1 >= 1.0 && a1 <= (double)p.S_w;  // false for NaN
    const bool integral = a0 == floor(a0) && a1 == floor(a1);
    if (p.err && !(in_range && integral)) atomicOr(p.err, (in_range ? 0 : AGYM_ERR_RES_RANGE) | (integral ? 0 : AGYM_ERR_RES_FRACTION));
    rh = min(max(in_range || a0 == a0 ? (int)fmin(fmax(a0, -1.0), 1.0e6) : 0, 1), p.S_h);
    rw = min(max(in_range || a1 == a1 ? (int)fmin(fmax(a1, -1.0), 1.0e6) : 0, 1), p.S_w);
}

// fov_loc update of the fixed fovea (fov_env.py:187-199), split into the global loads and the
// arithmetic so that a persistent kernel can issue the loads one env ahead.
struct LocIn {
    double a0, a1;
    int r, c, mode;
};

__device__ __forceinline__ LocIn load_loc_in(int n, const double *action, const uint8_t *ctrl, const int32_t *loc) {
    LocIn v;
    v.mode = ctrl ? ctrl[n] : AGYM_FOV_APPLY;
    v.r = loc[2 * n];
    v.c = loc[2 * n + 1];
    v.a0 = action ? action[2 * n] : 0.0;
    v.a1 = action ? action[2 * n + 1] : 0.0;
    return v;
}

__device__ __forceinline__ void apply_loc(const DevPlan &p, const LocIn &v, int &r, int &c) {
    r = v.r;
    c = v.c;
    if (v.mode == AGYM_FOV_RESET) {
        r = p.init_r;
        c = p.init_c;
    } else if (v.mode == AGYM_FOV_APPLY) {
        double a0 = v.a0, a1 = v.a1;
        if (p.relative) {
            a0 = (double)(r + clip_rint(a0, p.lo, p.hi));
            a1 = (double)(c + clip_rint(a1, p.lo, p.hi));
        }
        r = clip_rint(a0, 0.0, (double)(p.S_h - p.f_h));
        c = clip_rint(a1, 0.0, (double)(p.S_w - p.f_w));
    }
}

// STORE: write the new loc back (one thread per env); otherwise only compute it.
template <bool STORE = true>
__device__ __forceinline__ void update_loc_fixed(const DevPlan &p, int n, const double *action, const uint8_t *ctrl,
                                                 int32_t *loc, int &r, int &c) {
    apply_loc(p, load_loc_in(n, action, ctrl, loc), r, c);
    if (STORE) {
        loc[2 * n] = r;
        loc[2 * n + 1] = c;
    }
}

// ------------------------------------------------------------------ separable resamples
// dst[r][c] = sum_j w[c][j] * src[r][xmin[c] + j]      (pass along the contiguous axis)
template <typename SrcT>
__device__ __forceinline__ void resample_w(const SrcT *src, int sstride, float *dst, int dstride, int rows,
                                           const AxisRef &ax, int tid, int nt) {
    const int total = rows * ax.n_out;
    const FastDiv fd(ax.n_out);
    for (int i = tid; i < total; i += nt) {
        const int r = fd.div(i), c = i - r * ax.n_out;
        const SrcT *s = src + r * sstride + __ldg(ax.xmin + c);
        const float *w = ax.w + c * ax.taps;
        float acc = 0.f;
        for (int j = 0; j < ax.taps; ++j) acc = fmaf(__ldg(w + j), (float)s[j], acc);
        dst[r * dstride + c] = acc;
    }
}

// dst[r][c] = sum_j w[r][j] * src[xmin[r] + j][c]      (pass along the strided axis)
template <typename SrcT>
__device__ __forceinline__ void resample_h(const SrcT *src, int sstride, float *dst, int dstride, int cols,
                                           const AxisRef &ax, int tid, int nt) {
    const int total = ax.n_out * cols;
    const FastDiv fd(cols);
    for (int i = tid; i < total; i += nt) {
        const int r = fd.div(i), c = i - r * cols;
        const SrcT *s = src + __ldg(ax.xmin + r) * sstride + c;
        const float *w = ax.w + r * ax.taps;
        float acc = 0.f;
        for (int j = 0; j < ax.taps; ++j) acc = fmaf(__ldg(w + j), (float)s[j * sstride], acc);
        dst[r * dstride + c] = acc;
    }
}

// One output word (4 pixels of row y starting at column x0) of a strided-axis pass.
__device__ __forceinline__ uint32_t resample_h_word(const float *src, int sstride, const AxisRef &ax, int y, int x0) {
    const float *s = src + __ldg(ax.xmin + y) * sstride + x0;
    const float *w = ax.w + y * ax.taps;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int j = 0; j < ax.taps; ++j) {
        const float wj = __ldg(w + j);
        const float *sj = s + j * sstride;
        a0 = fmaf(wj, sj[0], a0);
        a1 = fmaf(wj, sj[1], a1);
        a2 = fmaf(wj, sj[2], a2);
        a3 = fmaf(wj, sj[3], a3);
    }
    return quant_u8(a0) | (quant_u8(a1) << 8) | (quant_u8(a2) << 16) | (quant_u8(a3) << 24);
}

// byte mask of the columns [c0, c1) inside the 4-byte word that starts at column x0
__device__ __forceinline__ uint32_t word_mask(int x0, int c0, int c1) {
    const int lo = max(c0 - x0, 0), hi = min(c1 - x0, 4);
    if (lo >= hi) return 0u;
    const uint32_t upto_hi = hi >= 4 ? 0xFFFFFFFFu : ((1u << (8 * hi)) - 1u);
    return upto_hi & ~((1u << (8 * lo)) - 1u);
}

// 16 interleaved 3-channel pixels (48 bytes, 12 words) -> 16 luma bytes.
// Y = (lw0 c0 + lw1 c1 + lw2 c2 + 16384) >> 15 (cv2's 15-bit luma, dmc_env.py:182) evaluated as
// (2 (lw . c) + 32768) >> 16, so that Y is byte 2 of the accumulator: one PRMT gathers a pixel's three
// bytes, two IDP.2A (16-bit weights x 8-bit channels) form the sum and PRMTs pack four results.
// w01 = 2 lw0 | 2 lw1 << 16, w2 = 2 lw2.
__device__ __forceinline__ uint4 luma16(const uint32_t (&w)[12], uint32_t w01, uint32_t w2) {
    uint32_t acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int j = 3 * i, wi = j >> 2, b = j & 3;  // compile time after unrolling
        // bytes b, b+1, b+2 of the pair (w[wi], w[wi + 1]); b <= 1 stays inside one word
        const uint32_t hi = wi + 1 < 12 ? w[wi + 1] : 0u;
        const uint32_t q = __byte_perm(w[wi], hi, (uint32_t)(b | (b + 1) << 4 | (b + 2) << 8 | 0x4000));
        acc[i] = __dp2a_hi(w2, q, __dp2a_lo(w01, q, 32768u));  // w2's upper half is 0: byte 3 of q does not matter
    }
    uint32_t o[4];
#pragma unroll
    for (int m = 0; m < 4; ++m)
        o[m] = __byte_perm(__byte_perm(acc[4 * m], acc[4 * m + 1], 0x0062), __byte_perm(acc[4 * m + 2], acc[4 * m + 3], 0x0062), 0x5410);
    return make_uint4(o[0], o[1], o[2], o[3]);
}

__device__ __forceinline__ size_t align16(size_t v) { return (v + 15) & ~size_t(15); }

// Two-tap expand of the cached squeeze (the peripheral kernels and the flexible fovea's peripheral background): lerp
// weights sum to one, so a bias of 49152.5 added in the W pass rides through both passes and the rounded pixel
// floor(v + 0.5) ends up in byte 1 of the float's bit pattern (ulp there is 2^-8, so the total evaluation error is
// < 0.01 u8 LSB) — no float->int conversion, one PRMT tree per 4 pixels.
constexpr float kBias = 49152.5f;

// Squeeze of one obs frame held in shared memory (u8) into the peripheral cache slot:
// Resize(peripheral_res) = W pass then H pass (fov_env.py:367).  Needs t1[S_h * p_w] floats.
__device__ void squeeze_to_cache(const DevPlan &p, const uint8_t *s_frame, float *s_t1, float *dst_global, int tid, int nt) {
    resample_w<uint8_t>(s_frame, p.S_w, s_t1, p.p_w, p.S_h, p.sq_w, tid, nt);
    __syncthreads();
    resample_h<float>(s_t1, p.p_w, dst_global, p.p_w, p.p_w, p.sq_h, tid, nt);
}

// ---- TMA (cp.async.bulk) + mbarrier helpers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
constexpr uint32_t kBackoffNs = 2000;  // suspend-time hint of the producer's try_wait
template <bool BACKOFF = false>
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        if (BACKOFF) {
            // a lone producer lane must not burn issue slots while it waits: let the hardware suspend
            // the thread on the barrier (suspend-time hint) instead of polling it
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(smem_u32(bar)), "r"(parity), "r"(kBackoffNs)
                : "memory");
        } else {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(smem_u32(bar)), "r"(parity)
                : "memory");
        }
    }
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// 4-D tiled tensor copy global -> shared through a CUtensorMap (TMA; SASS: UTMALDG), completing on an mbarrier
__device__ __forceinline__ void tensor_g2s_4d(void *smem_dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2, int c3) {
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}

// 1-D bulk copy shared -> global (TMA store; SASS: UBLKCP), tracked by bulk async-groups
__device__ __forceinline__ void bulk_s2g(void *gmem_dst, const void *smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// the issuing thread's bulk stores, all but the newest N groups, have finished READING shared memory
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// generic-proxy writes to shared memory become visible to the async proxy (TMA)
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// barrier among the consumer warps only (the producer warp never joins it)
__device__ __forceinline__ void consumer_sync() { asm volatile("bar.sync 1, %0;" ::"n"(kThreads) : "memory"); }
// barrier among the THREADS threads (whole warps) that share named barrier `id` (1..15; 0 is __syncthreads)
template <int THREADS>
__device__ __forceinline__ void named_sync(int id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(THREADS) : "memory"); }

// ---- programmatic dependent launch (PDL).  A kernel launched through launch_pdl() may start while the kernel before
// it in the stream is still draining: pdl_launch_dependents() (first statement of every such kernel) lets the NEXT
// kernel's CTAs be scheduled as soon as SM resources free up, and pdl_wait() — executed by every thread after the
// prologue that touches only the plan's constant tables and shared memory, and before the first access to any buffer a
// previous kernel may have written or may still read — blocks until the previous kernel has completed and flushed.
// What overlaps is launch latency, CTA ramp-up and the prologue; the data dependencies are unchanged.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- cp.async (LDGSTS) helpers
__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async16_s(uint32_t smem_addr, const void *gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async4_s(uint32_t smem_addr, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(gmem_src));
}
// 4-byte cp.async with compile-time byte offsets folded into the instruction's immediates
template <int SOFF, int GOFF>
__device__ __forceinline__ void cp_async4_imm(uint32_t smem_addr, const void *gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0 + %2], [%1 + %3], 4;" ::"r"(smem_addr), "l"(gmem_src), "n"(SOFF), "n"(GOFF));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- normalised second output (SURVEY.md section 8f row 3): the reference hands the agent float32(u) / 255
// (atari_env.py:75, dmc_env.py:183).  The observe kernels can write that value — as f32, or rounded once more to f16 /
// bf16 — next to the u8 observation, straight from the output words they already hold (no second pass over HBM).
// norm_u8: the correctly rounded quotient u / 255 by one FMA-corrected step on the reciprocal (q0 = u r, e = u - 255 q0
// exactly, q = q0 + e r); tests/test_gpu_parity.py compares all 256 values with the IEEE division of k_normalize.
__device__ __forceinline__ float norm_u8(uint32_t u) {
    const float x = (float)u, r = 1.0f / 255.0f;
    const float q0 = x * r;
    return fmaf(fmaf(-q0, 255.0f, x), r, q0);
}
// 4 pixels (one output word) -> dst[index]: 16 bytes of f32, or 8 bytes of f16 / bf16 (dt: AGYM_DTYPE_*)
__device__ __forceinline__ void norm_store4(int dt, uint32_t word, void *dst, size_t index) {
    const float f0 = norm_u8(word & 0xffu), f1 = norm_u8((word >> 8) & 0xffu), f2 = norm_u8((word >> 16) & 0xffu), f3 = norm_u8(word >> 24);
    if (dt == AGYM_DTYPE_F32) {
        reinterpret_cast<float4 *>(dst)[index] = make_float4(f0, f1, f2, f3);
    } else if (dt == AGYM_DTYPE_F16) {
        const __half2 a = __floats2half2_rn(f0, f1), b = __floats2half2_rn(f2, f3);
        reinterpret_cast<uint2 *>(dst)[index] = make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
    } else {
        const __nv_bfloat162 a = __floats2bfloat162_rn(f0, f1), b = __floats2bfloat162_rn(f2, f3);
        reinterpret_cast<uint2 *>(dst)[index] = make_uint2(*reinterpret_cast<const uint32_t *>(&a), *reinterpret_cast<const uint32_t *>(&b));
    }
}
// 16 pixels (four consecutive output words) -> dst vector `index` (64 bytes of f32, 32 bytes of f16 / bf16)
__device__ __forceinline__ void norm_store16(int dt, const uint4 v, void *dst, size_t index) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    if (dt == AGYM_DTYPE_F32) {
        float4 *o = reinterpret_cast<float4 *>(dst) + 4 * index;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            o[j] = make_float4(norm_u8(w[j] & 0xffu), norm_u8((w[j] >> 8) & 0xffu), norm_u8((w[j] >> 16) & 0xffu), norm_u8(w[j] >> 24));
    } else {
        uint32_t h[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float f0 = norm_u8(w[j] & 0xffu), f1 = norm_u8((w[j] >> 8) & 0xffu), f2 = norm_u8((w[j] >> 16) & 0xffu), f3 = norm_u8(w[j] >> 24);
            if (dt == AGYM_DTYPE_F16) {
                const __half2 a = __floats2half2_rn(f0, f1), b = __floats2half2_rn(f2, f3);
                h[2 * j] = *reinterpret_cast<const uint32_t *>(&a); h[2 * j + 1] = *reinterpret_cast<const uint32_t *>(&b);
            } else {
                const __nv_bfloat162 a = __floats2bfloat162_rn(f0, f1), b = __floats2bfloat162_rn(f2, f3);
                h[2 * j] = *reinterpret_cast<const uint32_t *>(&a); h[2 * j + 1] = *reinterpret_cast<const uint32_t *>(&b);
            }
        }
        uint4 *o = reinterpret_cast<uint4 *>(dst) + 2 * index;
        o[0] = make_uint4(h[0], h[1], h[2], h[3]);
        o[1] = make_uint4(h[4], h[5], h[6], h[7]);
    }
}

// ---- packed fp32 pairs (Blackwell FFMA2 / FADD2: two fp32 lanes per issue slot)
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, uint32_t &lo, uint32_t &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t fsub2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}

// ---- host-side launch helpers
template <typename F>
cudaError_t set_smem(F func, size_t bytes) {
    if (bytes > 48 * 1024)
        return cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    return cudaSuccess;
}

size_t a16(size_t v) { return (v + 15) & ~size_t(15); }

// AGYM_NO_PDL=1: plain stream-ordered launches (A/B comparisons)
const bool g_no_pdl = getenv("AGYM_NO_PDL") != nullptr;

// <<<grid, block, smem, st>>> with the programmatic-stream-serialization attribute (see pdl_wait above).  Only for
// kernels that execute pdl_wait() before their first dependent memory access.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = g_no_pdl ? 0 : 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);
}

// AGYM_NO_STD=1 forces the table-driven peripheral kernel even for the standard geometry
const bool g_disable_std = getenv("AGYM_NO_STD") != nullptr;
// AGYM_NO_TMA=1 forces the non-persistent ingest kernel (A/B comparisons, debugging)
const bool g_disable_tma = getenv("AGYM_NO_TMA") != nullptr;
// AGYM_FLEX_OLD=1 forces the one-CTA-per-env flexible kernel (A/B comparisons)
const bool g_flex_old = getenv("AGYM_FLEX_OLD") != nullptr;
// AGYM_CROP_OLD=1 forces the byte-gather crop kernel (A/B comparisons)
const bool g_crop_old = getenv("AGYM_CROP_OLD") != nullptr;
const bool g_crop_v2 = getenv("AGYM_CROP_V2") != nullptr;   // timing experiments: the round-2 crop kernel instead of v3
// AGYM_STD_NOFS=1: the standard-geometry peripheral kernel stages the fovea with per-thread 4-byte copies (A/B comparisons)
const bool g_std_nofs = getenv("AGYM_STD_NOFS") != nullptr;
// AGYM_INGEST_UNITS=n: units (shared-memory stages) per env of the TMA ingest kernel (tuning)
const int g_units = getenv("AGYM_INGEST_UNITS") ? atoi(getenv("AGYM_INGEST_UNITS")) : 0;


}  // namespace

}  // namespace agym
