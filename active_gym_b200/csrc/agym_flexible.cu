// sm_100a kernels: flexible fovea.
#include "agym_device.cuh"

namespace agym {

namespace {

// --------------------------------------------------------------------- observe: flexible
// FlexibleFovealEnv._fov_step + _get_fov_state (fov_env.py:270-330).
__device__ __forceinline__ AxisRef flex_axis(const DevPlan &p, int axis, int family, int r, int n_in) {
    const FlexEntry e = p.flex[(axis * 3 + family) * (p.S_max + 1) + r];
    AxisRef a;
    a.xmin = p.pool_i + e.xmin_off;
    a.w = reinterpret_cast<const float *>(p.pool_i + e.w_off);
    a.n_in = n_in; a.n_out = e.n_out; a.taps = e.taps;
    return a;
}

// Peripheral background of the flexible fovea, Resize(obs_size) of the cached squeeze (fov_env.py:366-368, 376): rows
// [y0, y1) of column quad q of one plane, from that plane's squeeze sq [p_h][p_w] and the plan's two-tap expand tables.
// The arithmetic is k_observe_peripheral_std's: W pass T = fma(w1, s[i0 + 1], fma(w0, s[i0], kBias)), H pass
// fma(w0, T[j] - T[j + 1], T[j + 1]), the pixel in byte 1 of the float; so the background is bit-identical to that
// kernel's at the standard geometry (its clamped border rows read T[0] twice: T[0] - T[1] and T[1] + (T[0] - T[1]) are
// exact, all T lying in [2^15, 2^16)).  dst: the word of row y0; rows are dstride words apart.
__device__ __forceinline__ void periph_expand(const DevPlan &p, const float *sq, int q, int y0, int y1, uint32_t *dst,
                                              int dstride) {
    int i0[4];
    float w0[4], w1[4], a[4], b[4];
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        i0[c] = __ldg(p.exw_i0 + 4 * q + c);
        w0[c] = __ldg(p.exw_w0 + 4 * q + c);
        w1[c] = __ldg(p.exw_w1 + 4 * q + c);
    }
    int j_have = -2;
    for (int y = y0; y < y1; ++y, dst += dstride) {
        const int j = __ldg(p.exh_i0 + y);
        const float wh = __ldg(p.exh_w0 + y);
        if (j != j_have) {   // squeezed rows j, j + 1 W-expanded (row j is the previous row j + 1 when the pair moves by one)
            const float *sa = sq + j * p.p_w, *sb = sa + p.p_w;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                a[c] = j == j_have + 1 ? b[c] : fmaf(w1[c], sa[i0[c] + 1], fmaf(w0[c], sa[i0[c]], kBias));
                b[c] = fmaf(w1[c], sb[i0[c] + 1], fmaf(w0[c], sb[i0[c]], kBias));
            }
            j_have = j;
        }
        uint32_t word = 0u;
#pragma unroll
        for (int c = 0; c < 4; ++c) word |= ((__float_as_uint(fmaf(wh, a[c] - b[c], b[c])) >> 8) & 0xffu) << (8 * c);
        *dst = word;
    }
}

// One plane of the table-driven kernel's peripheral variant: the window (bufA, rh x rw floats of its bytes), blurred iff
// rh > f_h in the arithmetic of the kernel that serves agym_observe_flexible(AGYM_OUT_MASK) on the same plan — the
// persistent kernel's 16-bit fixed-point W pass and fp32 H pass when the plan has those operators, the composed fp32
// operators of k_observe_flexible_fast otherwise — pasted onto the background of periph_expand (or, for expand tables
// that are not two-tap lerps, of k_observe_peripheral's generic passes).  Written byte by byte: out may sit at any address.
__device__ void periph_plane(const DevPlan &p, float *bufA, float *bufB, uint32_t *s_bg, const float *sq, int r0, int c0,
                             int rh, int rw, bool blur, uint8_t *out, int tid) {
    const FastDiv fd_rw(rw);
    if (blur) {
        const bool fixed_w = p.flexq != nullptr;
        const FlexEntry ew = fixed_w ? p.flexq[rw] : p.flexb[(p.S_max + 1) + rw];
        const FlexEntry eh = fixed_w ? p.flexh2[rh] : p.flexb[rh];
        for (int i = tid; i < rh * rw; i += kThreads) {   // W pass
            const int y = fd_rw.div(i), x = i - y * rw;
            const float *src = bufA + y * rw + __ldg(p.pool_i + ew.xmin_off + x);
            if (fixed_w) {   // flexq: {xmin, q16 weights in halves of 8 taps, halves, taps}
                const uint32_t *qw = reinterpret_cast<const uint32_t *>(p.pool_i + ew.w_off) + x * ew.taps * 4;
                uint32_t acc = 0u;
                for (int t = 0; t < ew.n_out; ++t) acc += ((__ldg(qw + (t >> 1)) >> (16 * (t & 1))) & 0xffffu) * (uint32_t)src[t];
                bufB[i] = (float)acc * (1.f / 65536.f);
            } else {
                const float *w = reinterpret_cast<const float *>(p.pool_i + ew.w_off) + x * ew.taps;
                float acc = 0.f;
                for (int t = 0; t < ew.taps; ++t) acc = fmaf(__ldg(w + t), src[t], acc);
                bufB[i] = acc;
            }
        }
        __syncthreads();
        const int wstep = fixed_w ? 2 : 1;   // flexh2 stores every weight twice
        for (int i = tid; i < rh * rw; i += kThreads) {   // H pass
            const int y = fd_rw.div(i), x = i - y * rw;
            const float *src = bufB + __ldg(p.pool_i + eh.xmin_off + y) * rw + x;
            const float *w = reinterpret_cast<const float *>(p.pool_i + eh.w_off) + wstep * y * eh.taps;
            float acc = 0.f;
            for (int t = 0; t < eh.taps; ++t) acc = fmaf(src[t * rw], __ldg(w + wstep * t), acc);
            bufA[i] = acc;
        }
    }
    const int quads = p.S_w >> 2;
    if (p.fast_expand) {
        const int nseg = min(p.S_h, max(1, kThreads / quads)), rows = (p.S_h + nseg - 1) / nseg;
        for (int i = tid; i < quads * nseg; i += kThreads) {
            const int g = i / quads, q = i - g * quads;
            periph_expand(p, sq, q, g * rows, min(p.S_h, g * rows + rows), s_bg + g * rows * quads + q, quads);
        }
    } else {   // squeeze -> s_sq, W pass -> s_t2, H pass per word (k_observe_peripheral<true>)
        float *s_sq = reinterpret_cast<float *>(s_bg + quads * p.S_h), *s_t2 = s_sq + p.p_h * p.p_w;
        for (int i = tid; i < p.p_h * p.p_w; i += kThreads) s_sq[i] = __ldg(sq + i);
        __syncthreads();
        resample_w<float>(s_sq, p.p_w, s_t2, p.S_w, p.p_h, p.ex_w, tid, kThreads);
        __syncthreads();
        for (int t = tid; t < quads * p.S_h; t += kThreads) {
            const int y = t / quads;
            s_bg[t] = resample_h_word(s_t2, p.S_w, p.ex_h, y, 4 * (t - y * quads));
        }
    }
    __syncthreads();
    const uint8_t *bg = reinterpret_cast<const uint8_t *>(s_bg);
    const FastDiv fd_sw(p.S_w);
    for (int i = tid; i < p.plane; i += kThreads) {   // fov_env.py:385-386 at the flexible window
        const int y = fd_sw.div(i), x = i - y * p.S_w;
        const int py = y - r0, px = x - c0;
        out[i] = (py >= 0 && py < rh && px >= 0 && px < rw) ? (uint8_t)quant_u8(bufA[py * rw + px]) : bg[i];
    }
    __syncthreads();
}

template <int VARIANT>
__global__ void __launch_bounds__(kThreads) k_observe_flexible(const __grid_constant__ DevPlan p,
                                                               const uint8_t *__restrict__ ring,
                                                               const int32_t *__restrict__ head,
                                                               const double *__restrict__ action,
                                                               const int32_t *__restrict__ atype,
                                                               const uint8_t *__restrict__ ctrl,
                                                               int32_t *__restrict__ loc, int32_t *__restrict__ res,
                                                               int pad_h, int pad_w, uint8_t *__restrict__ out,
                                                               const float *__restrict__ pcache) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_win[4];
    const int n = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        const int mode = ctrl ? ctrl[n] : AGYM_FOV_APPLY;
        int r = loc[2 * n], c = loc[2 * n + 1], rh = res[2 * n], rw = res[2 * n + 1];
        if (mode == AGYM_FOV_RESET) {
            r = p.init_r; c = p.init_c; rh = p.f_h; rw = p.f_w;
        } else if (mode == AGYM_FOV_APPLY) {
            const double a0 = action ? action[2 * n] : 0.0, a1 = action ? action[2 * n + 1] : 0.0;
            const int t = atype ? atype[n] : AGYM_ATYPE_FOV_LOC;
            if (t == AGYM_ATYPE_FOV_RES) {
                res_from_action(p, a0, a1, rh, rw);  // fov_res = action (fov_env.py:323)
                r = clip_rint((double)r, 0.0, (double)(p.S_h - rh));
                c = clip_rint((double)c, 0.0, (double)(p.S_w - rw));
            } else {
                double v0 = a0, v1 = a1;
                if (p.relative) {
                    v0 = (double)(r + clip_rint(a0, p.lo, p.hi));
                    v1 = (double)(c + clip_rint(a1, p.lo, p.hi));
                }
                r = clip_rint(v0, 0.0, (double)(p.S_h - rh));
                c = clip_rint(v1, 0.0, (double)(p.S_w - rw));
            }
        }
        loc[2 * n] = r; loc[2 * n + 1] = c; res[2 * n] = rh; res[2 * n + 1] = rw;
        s_win[0] = r; s_win[1] = c; s_win[2] = rh; s_win[3] = rw;
    }
    __syncthreads();
    const int r0 = s_win[0], c0 = s_win[1], rh = s_win[2], rw = s_win[3];
    const int h = head[n];
    const bool blur = rh > p.f_h;  // row dimension only (fov_env.py:286)

    float *bufA = reinterpret_cast<float *>(smem);
    float *bufB = bufA + p.plane;
    const FastDiv fd_rw(rw);
    const int oh = VARIANT == AGYM_OUT_CROP ? pad_h : p.S_h, ow = VARIANT == AGYM_OUT_CROP ? pad_w : p.S_w;
    const int oy = VARIANT == AGYM_OUT_MASK ? r0 : 0, ox = VARIANT == AGYM_OUT_MASK ? c0 : 0;
    const int wpr = ow / 4, wpp = oh * ow / 4;
    const FastDiv fd_wpr(wpr);

    for (int k = 0; k < p.K; ++k) {
        const uint8_t *src = ring + ((size_t)n * p.K + (h + 1 + k) % p.K) * p.plane;
        for (int i = tid; i < rh * rw; i += kThreads) {
            const int y = fd_rw.div(i), x = i - y * rw;
            bufA[i] = (float)__ldg(src + (r0 + y) * p.S_w + c0 + x);
        }
        __syncthreads();
        if constexpr (VARIANT == kOutPeriph) {
            periph_plane(p, bufA, bufB, reinterpret_cast<uint32_t *>(bufB + p.plane),
                         pcache + ((size_t)n * p.K + (h + 1 + k) % p.K) * p.p_h * p.p_w, r0, c0, rh, rw, blur,
                         out + ((size_t)n * p.K + k) * p.plane, tid);
            continue;
        }
        if (blur && VARIANT != AGYM_OUT_RESIZE_FOV) {  // Resize(fov_size) then Resize(fov_res) (fov_env.py:276-280)
            resample_w<float>(bufA, rw, bufB, p.f_w, rh, flex_axis(p, 1, 0, rw, rw), tid, kThreads);
            __syncthreads();
            resample_h<float>(bufB, p.f_w, bufA, p.f_w, p.f_w, flex_axis(p, 0, 0, rh, rh), tid, kThreads);
            __syncthreads();
            resample_w<float>(bufA, p.f_w, bufB, rw, p.f_h, flex_axis(p, 1, 1, rw, p.f_w), tid, kThreads);
            __syncthreads();
            resample_h<float>(bufB, rw, bufA, rw, rw, flex_axis(p, 0, 1, rh, p.f_h), tid, kThreads);
            __syncthreads();
        }
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)n * p.K + k) * oh * ow);
        if (VARIANT == AGYM_OUT_RESIZE_FOV) {
            // Resize(fov_size) of the unblurred window (fov_env.py:248,284-285), written byte by byte: a plane of
            // f_h * f_w bytes need not start on a word (the (21, 33) fovea, an output view at an odd address)
            resample_w<float>(bufA, rw, bufB, p.f_w, rh, flex_axis(p, 1, 0, rw, rw), tid, kThreads);
            __syncthreads();
            resample_h<float>(bufB, p.f_w, bufA, p.f_w, p.f_w, flex_axis(p, 0, 0, rh, rh), tid, kThreads);
            __syncthreads();
            uint8_t *d8 = out + ((size_t)n * p.K + k) * p.f_h * p.f_w;
            for (int i = tid; i < p.f_h * p.f_w; i += kThreads) d8[i] = (uint8_t)quant_u8(bufA[i]);
        } else if (VARIANT == AGYM_OUT_RESIZE_FULL) {
            resample_w<float>(bufA, rw, bufB, p.S_w, rh, flex_axis(p, 1, 2, rw, rw), tid, kThreads);
            __syncthreads();
            const AxisRef ah = flex_axis(p, 0, 2, rh, rh);
            for (int t = tid; t < wpp; t += kThreads) {
                const int y = fd_wpr.div(t), x0 = 4 * (t - y * wpr);
                dst[t] = resample_h_word(bufB, p.S_w, ah, y, x0);
            }
        } else {
            for (int t = tid; t < wpp; t += kThreads) {
                const int y = fd_wpr.div(t), x0 = 4 * (t - y * wpr);
                uint32_t word = 0u;
                const int py = y - oy;
                if (py >= 0 && py < rh) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int px = x0 + i - ox;
                        if (px >= 0 && px < rw) word |= quant_u8(bufA[py * rw + px]) << (8 * i);
                    }
                }
                dst[t] = word;
            }
        }
        __syncthreads();
    }
}

// Fast flexible fovea for the paste-type outputs (mask_out in place, or the zero-padded crop):
// the blur Resize(fov_size) -> Resize(fov_res) (fov_env.py:276-280) is applied as ONE banded operator
// per axis (host-composed, see build_blur_axis), i.e. two passes instead of four; the env's K windows
// are staged once as aligned words; the output frame is assembled in a shared-memory tile (zeros +
// window) and leaves as one TMA bulk store.
template <int VARIANT>
__global__ void __launch_bounds__(kThreads) k_observe_flexible_fast(const __grid_constant__ DevPlan p,
                                                                    const uint8_t *__restrict__ ring,
                                                                    const int32_t *__restrict__ head,
                                                                    const double *__restrict__ action,
                                                                    const int32_t *__restrict__ atype,
                                                                    const uint8_t *__restrict__ ctrl,
                                                                    int32_t *__restrict__ loc, int32_t *__restrict__ res,
                                                                    int oh, int ow, int t1_cap, uint8_t *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_win[4];
    const int n = blockIdx.x, tid = threadIdx.x;
    const int K = p.K, quads = p.S_w >> 2, xwm = quads + 1;
    const int tile_bytes = K * oh * ow;
    uint32_t *s_tile = reinterpret_cast<uint32_t *>(smem);                       // [K][oh][ow] bytes
    uint32_t *s_x = s_tile + (tile_bytes >> 2);                                  // [K][S_h][xwm] window words
    float *s_t1 = reinterpret_cast<float *>(s_x + K * p.S_h * xwm);              // [rh][rw]
    float *s_ww = s_t1 + t1_cap;                                                 // [S_w][blur_tmax]
    float *s_wh = s_ww + p.S_w * p.blur_tmax;                                    // [S_h][blur_tmax]
    int32_t *s_xw = reinterpret_cast<int32_t *>(s_wh + p.S_h * p.blur_tmax);     // [S_w] first tap
    int32_t *s_xh = s_xw + p.S_w;                                                // [S_h]
    if (tid == 0) {
        const int mode = ctrl ? ctrl[n] : AGYM_FOV_APPLY;
        int r = loc[2 * n], c = loc[2 * n + 1], rh = res[2 * n], rw = res[2 * n + 1];
        if (mode == AGYM_FOV_RESET) {
            r = p.init_r; c = p.init_c; rh = p.f_h; rw = p.f_w;
        } else if (mode == AGYM_FOV_APPLY) {
            const double a0 = action ? action[2 * n] : 0.0, a1 = action ? action[2 * n + 1] : 0.0;
            const int t = atype ? atype[n] : AGYM_ATYPE_FOV_LOC;
            if (t == AGYM_ATYPE_FOV_RES) {  // fov_res = action, then re-clamp loc (fov_env.py:322-324)
                res_from_action(p, a0, a1, rh, rw);
                r = clip_rint((double)r, 0.0, (double)(p.S_h - rh));
                c = clip_rint((double)c, 0.0, (double)(p.S_w - rw));
            } else {
                double v0 = a0, v1 = a1;
                if (p.relative) {
                    v0 = (double)(r + clip_rint(a0, p.lo, p.hi));
                    v1 = (double)(c + clip_rint(a1, p.lo, p.hi));
                }
                r = clip_rint(v0, 0.0, (double)(p.S_h - rh));
                c = clip_rint(v1, 0.0, (double)(p.S_w - rw));
            }
        }
        loc[2 * n] = r; loc[2 * n + 1] = c; res[2 * n] = rh; res[2 * n + 1] = rw;
        s_win[0] = r; s_win[1] = c; s_win[2] = rh; s_win[3] = rw;
    }
    {   // zero frame (everything outside the window stays zero)
        const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
        for (int i = tid; i < (tile_bytes >> 4); i += kThreads) reinterpret_cast<uint4 *>(s_tile)[i] = z4;
    }
    __syncthreads();
    const int r0 = s_win[0], c0 = s_win[1], rh = s_win[2], rw = s_win[3];
    const int h = head[n];
    const bool blur = rh > p.f_h;  // row dimension only (fov_env.py:286)
    const int oy = VARIANT == AGYM_OUT_MASK ? r0 : 0, ox = VARIANT == AGYM_OUT_MASK ? c0 : 0;
    // crop output may be narrower / shorter than the window only if the caller's pad is: clip
    const int vh = min(rh, oh - oy), vw = min(rw, ow - ox);

    // ---- stage the K windows as aligned words: row y of frame k at s_x[(k * S_h + y) * xwm ...]
    // (byte loads straight from the ring were measured 10 % slower)
    const int wq0 = c0 >> 2, nwx = ((c0 + rw - 1) >> 2) - wq0 + 1, cb = c0 & 3;
    {
        const uint32_t *ring_w = reinterpret_cast<const uint32_t *>(ring) + (size_t)n * K * (p.plane >> 2);
        const FastDiv fd_w(nwx), fd_h(rh);
        for (int i = tid; i < K * rh * nwx; i += kThreads) {
            const int row = fd_w.div(i), w = i - row * nwx;
            const int k = fd_h.div(row), y = row - k * rh;
            int slot = h + 1 + k;
            slot -= slot >= K ? K : 0;
            s_x[(k * p.S_h + y) * xwm + w] = __ldg(ring_w + (size_t)slot * (p.plane >> 2) + (r0 + y) * quads + wq0 + w);
        }
    }
    int tw = 1, th = 1;
    if (blur) {  // this env's two banded operators -> shared memory
        const FlexEntry ew = p.flexb[(p.S_max + 1) + rw], eh = p.flexb[rh];
        tw = ew.taps; th = eh.taps;
        const float *gw = reinterpret_cast<const float *>(p.pool_i + ew.w_off), *gh = reinterpret_cast<const float *>(p.pool_i + eh.w_off);
        for (int i = tid; i < rw * tw; i += kThreads) s_ww[i] = __ldg(gw + i);
        for (int i = tid; i < rh * th; i += kThreads) s_wh[i] = __ldg(gh + i);
        for (int i = tid; i < rw; i += kThreads) s_xw[i] = __ldg(p.pool_i + ew.xmin_off + i);
        for (int i = tid; i < rh; i += kThreads) s_xh[i] = __ldg(p.pool_i + eh.xmin_off + i);
    }
    __syncthreads();
    const uint8_t *xb = reinterpret_cast<const uint8_t *>(s_x) + cb;
    uint8_t *tb = reinterpret_cast<uint8_t *>(s_tile);
    const FastDiv fd_rw(rw);
    if (!blur) {  // the window itself, bit exact
        const FastDiv fd_rh(rh);
        for (int i = tid; i < K * rh * rw; i += kThreads) {
            const int row = fd_rw.div(i), x = i - row * rw;
            const int k = fd_rh.div(row), y = row - k * rh;
            if (y < vh && x < vw) tb[(k * oh + oy + y) * ow + ox + x] = xb[((k * p.S_h + y) * xwm) * 4 + x];
        }
    } else {
        // t1 rows are padded to a multiple of 4 floats so that the H pass reads float4; as many frames
        // per pass as fit (all K for windows up to ~50 x 52), so an env costs 2 barriers instead of 2K
        const int rwp = (rw + 3) & ~3, per = rh * rwp;
        const int kg = K * per <= t1_cap ? K : 1;
        const FastDiv fd_fr(rh * rw), fd_q(rwp >> 2), fd_frq(rh * (rwp >> 2));
        for (int k0 = 0; k0 < K; k0 += kg) {
            // W pass: t1[y][x] = sum_t Mw[x][t] * X[y][xw[x] + t]
            for (int i = tid; i < kg * rh * rw; i += kThreads) {
                const int kk = fd_fr.div(i), rem = i - kk * rh * rw;
                const int y = fd_rw.div(rem), x = rem - y * rw;
                const uint8_t *src = xb + (((k0 + kk) * p.S_h + y) * xwm) * 4 + s_xw[x];
                const float *w = s_ww + x * tw;
                float acc = 0.f;
                for (int t = 0; t < tw; ++t) acc = fmaf(w[t], (float)src[t], acc);
                s_t1[kk * per + y * rwp + x] = acc;
            }
            __syncthreads();
            // H pass, 4 columns per thread + quantise + paste: out[y][x] = sum_t Mh[y][t] * t1[xh[y] + t][x]
            for (int i = tid; i < kg * rh * (rwp >> 2); i += kThreads) {
                const int kk = fd_frq.div(i), rem = i - kk * rh * (rwp >> 2);
                const int y = fd_q.div(rem), x0 = 4 * (rem - y * (rwp >> 2));
                const float *src = s_t1 + kk * per + s_xh[y] * rwp + x0;
                const float *w = s_wh + y * th;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int t = 0; t < th; ++t) {
                    const float4 v = *reinterpret_cast<const float4 *>(src + t * rwp);
                    const float wt = w[t];
                    acc.x = fmaf(wt, v.x, acc.x); acc.y = fmaf(wt, v.y, acc.y);
                    acc.z = fmaf(wt, v.z, acc.z); acc.w = fmaf(wt, v.w, acc.w);
                }
                if (y < vh) {
                    uint8_t *o = tb + ((k0 + kk) * oh + oy + y) * ow + ox + x0;
                    if (x0 < vw) o[0] = (uint8_t)quant_u8(acc.x);
                    if (x0 + 1 < vw) o[1] = (uint8_t)quant_u8(acc.y);
                    if (x0 + 2 < vw) o[2] = (uint8_t)quant_u8(acc.z);
                    if (x0 + 3 < vw) o[3] = (uint8_t)quant_u8(acc.w);
                }
            }
            __syncthreads();
        }
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
        bulk_s2g(out + (size_t)n * tile_bytes, s_tile, (uint32_t)tile_bytes);
        bulk_commit();
        bulk_wait_read<0>();
    }
}

// Persistent flexible fovea (mask_out in place, or the zero-padded crop): the successor of
// k_observe_flexible_fast.  Two CTAs per SM pull envs from a device counter (windows of 20..50 pixels,
// blurred or not, make an env's cost vary 3x: a static split left a quarter of the SM time idle) and
// keep three things in flight:
//   * thread 0 claims the env two iterations ahead and applies its sensory action (fov_env.py:314-330):
//     the atomic, the loads and the arithmetic are spread over the phases of the current env;
//   * the K windows of the next env (and its W operator) travel by cp.async during the current H pass;
//   * the finished frame tile leaves as one TMA bulk store while the next env is computed.
// The blur Resize(fov_size) -> Resize(fov_res) (fov_env.py:276-280) is one banded operator per axis.
// Along W it runs on the staged bytes in 16-bit fixed point: 8 taps = 4 IDP.2A on a funnel-shifted
// 8-byte window, two rows per thread, weights * 2^16 summing to 2^16 exactly (<= 255 * taps / 2^17 LSB
// from the fp64 weights: 0.01 LSB for the 5-tap operators of windows up to 50).  Along H it is packed
// fp32 (FFMA2) on four columns per thread; results are rounded to nearest-even with the 1.5 * 2^23 bias
// and leave as whole words.
// VARIANT AGYM_OUT_RESIZE_FOV (the glimpse, Resize(fov_size) of the unblurred window, fov_env.py:248,284-285) reuses
// the claims, the fov update, the strip copies and the operator prefetch; its two passes (rw -> f_w, then rh -> f_h)
// are fp32 with the r -> f tables of family 0, evaluated in the order of the table-driven kernel (bit-identical to it).
// The tile is K * f_h * f_w bytes with no zero fill; a tile that is not a multiple of 16 bytes (f_w = 30 at K = 3 or
// K * C = 9) or a 16-byte-misaligned output leaves as 4-byte words from the worker threads instead of the bulk store.
// VARIANT kOutPeriph (agym_observe_flexible_peripheral) is mask_out over the peripheral background: the env's K-plane
// squeeze (contiguous in pcache) arrives with the strips on the same mbarrier, the workers expand it into the tile where
// mask_out zero-fills (periph_expand), and both paste paths merge the first / last word of every window row into that
// background (FlexGeom::m_first / m_last) instead of overwriting its bytes with zeros.
#ifndef AGYM_FLEX_THREADS
#define AGYM_FLEX_THREADS 256
#endif
constexpr int kFlexThreads = AGYM_FLEX_THREADS;


struct FlexGeom {
    int rh, rwp, vh, nq, ow4, oh, wlo, oy;
    uint32_t m_first, m_last;  // byte masks of the first / last output word of a window row
};

// H pass over kc frames (MERGE: over a background instead of zeros).  A thread OWNS an output word (window row y, word q): the row's weights, its first source row
// and the word's byte mask stay in registers while the thread walks through the kc frames (pointer increments only) —
// 25 instead of 70 instructions per output word for a 5-tap row.  s_wh2 holds every weight twice (FFMA2 operand).
template <int TH, bool MERGE>
__device__ __forceinline__ void flex_hpass(const FlexGeom &g, const float *s_t1, const uint64_t *s_wh2, const int32_t *s_xh,
                                           uint32_t *s_tile, int k0, int kc, int th, int tid, const uint32_t *s_magic) {
    const FastDiv fd_nq(g.nq, s_magic);
    const int pairs = g.vh * g.nq;                        // rows past the frame's edge (y >= vh) produce nothing
    const int fstride = g.rh * g.rwp, tstride = g.oh * g.ow4;
    const uint64_t rne2 = pack2(12582912.f, 12582912.f);  // 1.5 * 2^23: v + bias has rint(v) (half to even) in its low byte
    for (int pr = tid; pr < pairs; pr += kFlexThreads) {
        const int y = fd_nq.div(pr), q = pr - y * g.nq;
        const float *src = s_t1 + s_xh[y] * g.rwp + 4 * q;
        uint32_t *dst = s_tile + (k0 * g.oh + g.oy + y) * g.ow4 + g.wlo + q;
        uint32_t mask = 0xffffffffu;
        if (q == 0) mask &= g.m_first;
        if (q == g.nq - 1) mask &= g.m_last;
        const uint64_t *w = s_wh2 + y * th;
        uint64_t wr[TH > 0 ? TH : 1];
        if (TH > 0) {
#pragma unroll
            for (int t = 0; t < TH; ++t) wr[t] = w[t];
        }
        for (int kk = 0; kk < kc; ++kk, src += fstride, dst += tstride) {
            uint64_t a01 = 0ull, a23 = 0ull;
            if (TH > 0) {
#pragma unroll
                for (int t = 0; t < TH; ++t) {
                    const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(src + t * g.rwp);
                    a01 = ffma2(v.x, wr[t], a01);
                    a23 = ffma2(v.y, wr[t], a23);
                }
            } else {
                for (int t = 0; t < th; ++t) {
                    const ulonglong2 v = *reinterpret_cast<const ulonglong2 *>(src + t * g.rwp);
                    const uint64_t wt = w[t];
                    a01 = ffma2(v.x, wt, a01);
                    a23 = ffma2(v.y, wt, a23);
                }
            }
            uint32_t b0, b1, b2, b3;
            unpack2(fadd2(a01, rne2), b0, b1);
            unpack2(fadd2(a23, rne2), b2, b3);
            const uint32_t v = __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410) & mask;
            *dst = MERGE ? (*dst & ~mask) | v : v;   // MERGE: the edge words keep the background's bytes
        }
    }
}

// W pass over nrows staged rows: t1[row][sb + x] = 2^-16 * sum_t q[x][t] * X[row][xw[x] + t].  A thread OWNS output
// column x (its weights, first tap and shift stay in registers for the whole env) and walks down the rows of its row
// group, two rows per iteration (two independent IDP.2A chains): 28 instructions per two outputs instead of the 57 of
// the item-per-iteration form, whose index arithmetic and weight reloads were a quarter of the kernel (ncu source view).
// The staged rows are the full-width strips of the K frames (strip_w words apart, rows row_w words apart; xrow0 = the
// first window row of frame k0, c0 = the window's first column): row r of the group is row r % rh of frame r / rh.
template <int NH>
__device__ __forceinline__ void flex_wpass(const uint32_t *xrow0, int rh, int row_w, int strip_w, const int32_t *s_xw, const uint32_t *s_wq,
                                           float *s_t1, int rwp, int sb, int c0, int rw, int nrows, int tid, const uint32_t *s_magic) {
    const FastDiv fd_rw(rw, s_magic), fd_rh(rh, s_magic);
    const int kfix = strip_w - rh * row_w;
    const int G = fd_rw.div(kFlexThreads);           // row groups: kFlexThreads / rw >= 3 (rw <= 84)
    const int g = fd_rw.div(tid), x = tid - g * rw;
    if (g >= G) return;                              // the kFlexThreads - G * rw threads past the last group
    const int b = c0 + s_xw[x];
    const uint32_t sh = (uint32_t)(b & 3) * 8u;
    uint4 q[NH];
#pragma unroll
    for (int hh = 0; hh < NH; ++hh) q[hh] = reinterpret_cast<const uint4 *>(s_wq)[x * NH + hh];
    const uint32_t *sp0 = xrow0 + (b >> 2);
    float *d = s_t1 + g * rwp + sb + x;
    const int step_d = G * rwp;
    for (int r = g; r < nrows; r += 2 * G, d += 2 * step_d) {
        const bool two = r + G < nrows;
        const int r1 = two ? r + G : r;                  // the second row of the iteration (the first again past the end)
        const uint32_t *sp = sp0 + r * row_w + fd_rh.div(r) * kfix;
        const uint32_t *sp1 = sp0 + r1 * row_w + fd_rh.div(r1) * kfix;
        uint32_t acc0 = 0u, acc1 = 0u;
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
            const uint32_t a0 = sp[2 * hh], a1 = sp[2 * hh + 1], a2 = sp[2 * hh + 2];
            const uint32_t c0 = sp1[2 * hh], c1 = sp1[2 * hh + 1], c2 = sp1[2 * hh + 2];
            const uint32_t lo0 = __funnelshift_r(a0, a1, sh), hi0 = __funnelshift_r(a1, a2, sh);
            const uint32_t lo1 = __funnelshift_r(c0, c1, sh), hi1 = __funnelshift_r(c1, c2, sh);
            acc0 = __dp2a_lo(q[hh].x, lo0, acc0); acc0 = __dp2a_hi(q[hh].y, lo0, acc0);
            acc1 = __dp2a_lo(q[hh].x, lo1, acc1); acc1 = __dp2a_hi(q[hh].y, lo1, acc1);
            acc0 = __dp2a_lo(q[hh].z, hi0, acc0); acc0 = __dp2a_hi(q[hh].w, hi0, acc0);
            acc1 = __dp2a_lo(q[hh].z, hi1, acc1); acc1 = __dp2a_hi(q[hh].w, hi1, acc1);
        }
        d[0] = (float)acc0 * (1.f / 65536.f);
        if (two) d[step_d] = (float)acc1 * (1.f / 65536.f);
    }
}

// Glimpse W pass over nrows staged rows (row r = row r % rh of frame r / rh): t1[r][x] = sum_t w[x][t] * X[r][c0 + xw[x] + t]
// for the f_w output columns, fp32 in the tap order of resample_w.
__device__ __forceinline__ void glimpse_wpass(const uint32_t *xrow0, int rh, int S_w, int strip_w, const int32_t *s_xw,
                                              const float *s_ww, int tw, float *s_t1, int f_w, int c0, int nrows, int tid,
                                              const uint32_t *s_magic) {
    const FastDiv fd_fw(f_w, s_magic), fd_rh(rh, s_magic);
    for (int i = tid; i < nrows * f_w; i += kFlexThreads) {
        const int row = fd_fw.div(i), x = i - row * f_w;
        const int kk = fd_rh.div(row), y = row - kk * rh;
        const uint8_t *src = reinterpret_cast<const uint8_t *>(xrow0 + kk * strip_w) + y * S_w + c0 + s_xw[x];
        const float *w = s_ww + x * tw;
        float acc = 0.f;
        for (int t = 0; t < tw; ++t) acc = fmaf(w[t], (float)src[t], acc);
        s_t1[i] = acc;
    }
}

// Glimpse H pass over nfr frames of t1 (rh x f_w each): tile byte (k, y, x) = rint(sum_t w[y][t] * t1[k][xh[y] + t][x]),
// fp32 in the tap order of resample_h.  Output index i is the tile's byte offset: words straddle rows at f_w = 30.
__device__ __forceinline__ void glimpse_hpass(const float *s_t1, int rh, const int32_t *s_xh, const float *s_wh, int th,
                                              uint8_t *tb, int f_h, int f_w, int nfr, int tid, const uint32_t *s_magic) {
    const FastDiv fd_fw(f_w, s_magic), fd_fh(f_h, s_magic);
    for (int i = tid; i < nfr * f_h * f_w; i += kFlexThreads) {
        const int row = fd_fw.div(i), x = i - row * f_w;
        const int kk = fd_fh.div(row), y = row - kk * f_h;
        const float *src = s_t1 + (kk * rh + s_xh[y]) * f_w + x;
        const float *w = s_wh + y * th;
        float acc = 0.f;
        for (int t = 0; t < th; ++t) acc = fmaf(w[t], src[t * f_w], acc);
        tb[i] = (uint8_t)quant_u8(acc);
    }
}

template <int VARIANT>
__global__ void __launch_bounds__(kFlexThreads + 32, 2) k_observe_flexible_v3(const __grid_constant__ DevPlan p,
                                                                          const uint8_t *__restrict__ ring,
                                                                          const int32_t *__restrict__ head,
                                                                          const double *__restrict__ action,
                                                                          const int32_t *__restrict__ atype,
                                                                          const uint8_t *__restrict__ ctrl,
                                                                          int32_t *__restrict__ loc, int32_t *__restrict__ res,
                                                                          int oh, int ow, int t1_cap, uint8_t *__restrict__ out,
                                                                          int *__restrict__ counters, int word_store,
                                                                          const float *__restrict__ pcache) {
    extern __shared__ __align__(16) uint8_t smem[];
    constexpr int kWin = 4;
    constexpr bool kPeriph = VARIANT == kOutPeriph;   // the window pasted onto the peripheral background
    // per claimed env: index, window, ring head, and where its operators live in the pool
    __shared__ int s_en[kWin], s_er[kWin], s_ec[kWin], s_erh[kWin], s_erw[kWin], s_ehd[kWin];
    __shared__ int s_eth[kWin], s_ehw[kWin], s_ehx[kWin], s_enh[kWin], s_eqw[kWin], s_eqx[kWin];
    __shared__ uint32_t s_magic[256];              // FastDiv multipliers of 1..255: a division per divisor and env otherwise
    __shared__ __align__(8) uint64_t s_bar;        // completion of an env's K strip copies (phase = env count & 1)
    const int tid = threadIdx.x;
    if (tid < 256) s_magic[tid] = tid ? 0xFFFFFFFFu / (uint32_t)tid + 1u : 0u;
    if (tid == kFlexThreads) { mbar_init(&s_bar, 1); mbar_fence_init(); }
    const bool worker = tid < kFlexThreads;        // warps 0 .. 7/11 compute, the last warp is the control warp
    const bool boss = tid == kFlexThreads;         // its lane 0: env claims, fov updates, TMA stores
    const int K = p.K, quads = p.S_w >> 2, xcap = quads + 2, strip_w = (p.plane + 16) >> 2;
    const int tile_bytes = K * oh * ow;
    uint32_t *s_tile = reinterpret_cast<uint32_t *>(smem);                          // [K][oh][ow] bytes
    uint32_t *s_x = reinterpret_cast<uint32_t *>(smem + align16((size_t)tile_bytes));  // [K][strip_w]: the windows' full-width row strips
    const int pp = p.p_h * p.p_w, sq_bytes = kPeriph ? 4 * K * pp : 0;
    const size_t o_sq = align16(align16((size_t)tile_bytes) + 4 * (size_t)K * p.S_h * xcap);
    float *s_sq = reinterpret_cast<float *>(smem + o_sq);                          // kPeriph: [K slots][p_h][p_w] squeeze
    float *s_t1 = reinterpret_cast<float *>(smem + align16(o_sq + sq_bytes));     // [kg * rh][rwp]
    uint32_t *s_wq = reinterpret_cast<uint32_t *>(s_t1 + t1_cap);                   // [rw][halves][4]; t1_cap % 4 == 0
    uint64_t *s_wh2 = reinterpret_cast<uint64_t *>(s_wq + p.S_w * 8);               // [rh][th] {w, w}
    int32_t *s_xw = reinterpret_cast<int32_t *>(s_wh2 + p.S_h * p.blur_tmax);       // [rw] first tap
    int32_t *s_xh = s_xw + p.S_w;                                                   // [rh]
    const int N = p.N;

    // ---- boss: claim an env, load what its fov update needs, apply it (three steps, spread over an iteration)
    struct Pend { int n, mode, r, c, rh, rw, hd, t; double a0, a1; };
    // envs blockIdx.x and blockIdx.x + G are this CTA's without asking; the counter hands out the rest.  A claim
    // is only issued here: its value is looked at a barrier later, so nobody waits for the atomic's round trip
    bool more = true;
    const int n_static = 2 * (int)gridDim.x;
    auto claim = [&]() { return more ? n_static + atomicAdd(counters, 1) : N; };
    auto load_env = [&](int n, Pend &q) {
        q.n = n;
        if (n >= N) return;
        q.mode = ctrl ? ctrl[n] : AGYM_FOV_APPLY;
        q.r = loc[2 * n]; q.c = loc[2 * n + 1]; q.rh = res[2 * n]; q.rw = res[2 * n + 1];
        q.hd = head[n];
        q.a0 = action ? action[2 * n] : 0.0; q.a1 = action ? action[2 * n + 1] : 0.0;
        q.t = atype ? atype[n] : AGYM_ATYPE_FOV_LOC;
    };
    auto finish_env = [&](const Pend &q, int e) {
        s_en[e] = q.n;
        if (q.n >= N) return;
        int r = q.r, c = q.c, rh = q.rh, rw = q.rw;
        double a0 = q.a0, a1 = q.a1;
        // the control thread's fp64 chain must stay inside its branch: without this fence the compiler speculates the
        // ~60 fp64 instructions above `if (boss)` and every warp executes them for every env (ncu source view)
        asm volatile("" : "+d"(a0), "+d"(a1), "+r"(r), "+r"(c));
        if (q.mode == AGYM_FOV_RESET) {
            r = p.init_r; c = p.init_c; rh = p.f_h; rw = p.f_w;
        } else if (q.mode == AGYM_FOV_APPLY) {
            if (q.t == AGYM_ATYPE_FOV_RES) {  // fov_res = action, then re-clamp loc (fov_env.py:322-324)
                res_from_action(p, a0, a1, rh, rw);
                r = clip_rint((double)r, 0.0, (double)(p.S_h - rh));
                c = clip_rint((double)c, 0.0, (double)(p.S_w - rw));
            } else {
                double v0 = a0, v1 = a1;
                if (p.relative) {
                    v0 = (double)(r + clip_rint(a0, p.lo, p.hi));
                    v1 = (double)(c + clip_rint(a1, p.lo, p.hi));
                }
                r = clip_rint(v0, 0.0, (double)(p.S_h - rh));
                c = clip_rint(v1, 0.0, (double)(p.S_w - rw));
            }
        }
        const int n = q.n;
        loc[2 * n] = r; loc[2 * n + 1] = c; res[2 * n] = rh; res[2 * n + 1] = rw;
        s_er[e] = r; s_ec[e] = c; s_erh[e] = rh; s_erw[e] = rw; s_ehd[e] = q.hd;
        if constexpr (VARIANT == AGYM_OUT_RESIZE_FOV) {   // r -> f on both axes (family 0)
            const FlexEntry eh = p.flex[rh], ew = p.flex[3 * (p.S_max + 1) + rw];
            s_eth[e] = eh.taps; s_ehw[e] = eh.w_off; s_ehx[e] = eh.xmin_off;
            s_enh[e] = ew.taps; s_eqw[e] = ew.w_off; s_eqx[e] = ew.xmin_off;
        } else if (rh > p.f_h) {
            const FlexEntry eh = p.flexh2[rh], ew = p.flexq[rw];
            s_eth[e] = eh.taps; s_ehw[e] = eh.w_off; s_ehx[e] = eh.xmin_off;
            s_enh[e] = ew.taps; s_eqw[e] = ew.w_off; s_eqx[e] = ew.xmin_off;
        }
    };
    // ---- boss: the K windows of entry e as the full-width strips of their rows, one TMA bulk copy per frame (a strip is
    // contiguous in the ring; its 16-byte-aligned hull starts `lead` bytes early, the same for every frame because a
    // plane is a multiple of 16 bytes).  No thread spends instructions on the windows; the strips complete on s_bar.
    auto fetch_strips = [&](int e) {
        const int n = s_en[e];
        if (n >= N) return;
        const int r0 = s_er[e], rh = s_erh[e], h = s_ehd[e];
        const uint32_t first = (uint32_t)(r0 * p.S_w), lead = first & 15u;
        const uint32_t bytes = (lead + (uint32_t)(rh * p.S_w) + 15u) & ~15u;
        const uint8_t *src = ring + (size_t)n * K * p.plane + (first - lead);
        mbar_expect_tx(&s_bar, bytes * (uint32_t)K + (uint32_t)sq_bytes);
        if (kPeriph) bulk_g2s(s_sq, pcache + (size_t)n * K * pp, (uint32_t)sq_bytes, &s_bar);   // the env's K slots, contiguous
        for (int k = 0; k < K; ++k) {
            int slot = h + 1 + k;
            slot -= slot >= K ? K : 0;
            bulk_g2s(s_x + k * strip_w, src + (size_t)slot * p.plane, bytes, &s_bar);
        }
    };
    // ---- workers: the W operator of entry e by cp.async (one group)
    auto prefetch = [&](int e) {
        const int n = s_en[e];
        if constexpr (VARIANT == AGYM_OUT_RESIZE_FOV) {   // f_w rows of fp32 weights (the pool is only 4-byte aligned)
            if (n < N) {
                const int32_t *gq = p.pool_i + s_eqw[e], *gx = p.pool_i + s_eqx[e];
                for (int i = tid; i < p.f_w * s_enh[e]; i += kFlexThreads) cp_async4(s_wq + i, gq + i);
                for (int i = tid; i < p.f_w; i += kFlexThreads) cp_async4(s_xw + i, gx + i);
            }
        } else if (n < N && s_erh[e] > p.f_h) {
            const int rw = s_erw[e];
            const int32_t *gq = p.pool_i + s_eqw[e], *gx = p.pool_i + s_eqx[e];
            for (int i = tid; i < rw * s_enh[e]; i += kFlexThreads) cp_async16(s_wq + 4 * i, gq + 4 * i);
            for (int i = tid; i < rw; i += kFlexThreads) cp_async4(s_xw + i, gx + i);
        }
        cp_async_commit();
    };

    // kPeriph: background items (frame, row segment, column quad), nseg segments of `rows` rows per plane, chosen for
    // the fewest rows per worker thread (3 x 28 rows at K = 4, 4 x 21 at K = 3 and K * C = 9)
    int nseg = 1, rows = p.S_h;
    if (kPeriph) {
        for (int sg = 1, best = 1 << 30; sg <= 8; ++sg) {
            const int cost = ((K * quads * sg + kFlexThreads - 1) / kFlexThreads) * ((p.S_h + sg - 1) / sg);
            if (cost < best) { best = cost; nseg = sg; }
        }
        rows = (p.S_h + nseg - 1) / nseg;
    }
    if (boss) {
        Pend q0, q1;
        load_env(min((int)blockIdx.x, N), q0);
        load_env(min((int)(blockIdx.x + gridDim.x), N), q1);
        finish_env(q0, 0);
        finish_env(q1, 1);
        more = q1.n < N;
        fetch_strips(0);
    }
    __syncthreads();
    if (worker) prefetch(0);

    for (int j = 0;; ++j) {
        const int e = j & (kWin - 1), n = s_en[e];
        if (n >= N) break;
        int n2 = N;
        if (boss) n2 = claim();                  // the env two iterations ahead; the result is not needed before #1
        const int r0 = s_er[e], c0 = s_ec[e], rh = s_erh[e], rw = s_erw[e];
        const bool blur = rh > p.f_h;  // row dimension only (fov_env.py:286)
        const int oy = VARIANT == AGYM_OUT_MASK || kPeriph ? r0 : 0, ox = VARIANT == AGYM_OUT_MASK || kPeriph ? c0 : 0;
        const int cb = c0 & 3, sb = ox & 3;
        const int vw = min(rw, ow - ox);
        FlexGeom g;
        g.rh = rh; g.oy = oy; g.oh = oh; g.ow4 = ow >> 2; g.wlo = ox >> 2;
        g.vh = min(rh, oh - oy);
        g.nq = ((sb + vw - 1) >> 2) + 1;
        g.rwp = (sb + rw + 3) & ~3;
        g.m_first = word_mask(0, sb, sb + vw);
        g.m_last = word_mask(4 * (g.nq - 1), sb, sb + vw);
        const uint32_t *s_xs = s_x + ((r0 * p.S_w & 15) >> 2);   // first window row of frame 0 (behind the hull's lead)
        int th = 1, nh = 1;
        if constexpr (VARIANT == AGYM_OUT_RESIZE_FOV) {   // this env's H operator (f_h rows), as below
            th = s_eth[e];
            nh = s_enh[e];
            if (worker) {
                const int32_t *gh = p.pool_i + s_ehw[e], *gx = p.pool_i + s_ehx[e];
                for (int i = tid; i < p.f_h * th; i += kFlexThreads) cp_async4(reinterpret_cast<float *>(s_wh2) + i, gh + i);
                for (int i = tid; i < p.f_h; i += kFlexThreads) cp_async4(s_xh + i, gx + i);
            }
        } else if (blur) {  // this env's H operator; s_wh2 / s_xh were last read before the previous env's final barrier
            th = s_eth[e];
            nh = s_enh[e];
            if (worker) {
                const int32_t *gh = p.pool_i + s_ehw[e], *gx = p.pool_i + s_ehx[e];
                for (int i = tid; i < (rh * th + 1) >> 1; i += kFlexThreads) cp_async16(s_wh2 + 2 * i, gh + 4 * i);
                for (int i = tid; i < rh; i += kFlexThreads) cp_async4(s_xh + i, gx + i);
            }
        }
        cp_async_commit();
        cp_async_wait<1>();                    // this thread's part of the W operator has landed
        if (worker) mbar_wait(&s_bar, (uint32_t)j & 1u);   // the strips of this env (the j-th of this CTA) have landed
        if (boss) bulk_wait_read<0>();         // the previous tile has been read by the TMA store
        __syncthreads();                       // #1
        Pend pend;
        pend.n = N;
        if (boss) {
            if (n2 >= N) { n2 = N; more = false; }
            load_env(n2, pend);
        }
        if (worker && kPeriph) {   // the background: every plane expanded from its squeeze (s_sq is refilled after #2)
            const FastDiv fd_q(quads, s_magic), fd_s(nseg, s_magic);
            for (int i = tid; i < K * nseg * quads; i += kFlexThreads) {
                const int rest = fd_q.div(i), q = i - rest * quads;
                const int kk = fd_s.div(rest), y0 = (rest - kk * nseg) * rows;
                int slot = s_ehd[e] + 1 + kk;
                slot -= slot >= K ? K : 0;
                periph_expand(p, s_sq + slot * pp, q, y0, min(p.S_h, y0 + rows), s_tile + (kk * p.S_h + y0) * quads + q, quads);
            }
        } else if (worker && VARIANT != AGYM_OUT_RESIZE_FOV) {   // zero frame (everything outside the window stays zero)
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            for (int i = tid; i < (tile_bytes >> 4); i += kFlexThreads) reinterpret_cast<uint4 *>(s_tile)[i] = z4;
        }
        const int per = VARIANT == AGYM_OUT_RESIZE_FOV ? rh * ow : blur ? rh * g.rwp : rh * g.nq;
        const int kg = min(K, t1_cap / per);
        for (int k0 = 0; k0 < K; k0 += kg) {
            const int kc = min(kg, K - k0);
            const bool last = k0 + kc >= K;
            if (k0) __syncthreads();           // the previous group's H pass has read t1
            if (!worker) {
            } else if (VARIANT == AGYM_OUT_RESIZE_FOV) {
                glimpse_wpass(s_xs + k0 * strip_w, rh, p.S_w, strip_w, s_xw, reinterpret_cast<const float *>(s_wq), nh, s_t1, ow, c0,
                              kc * rh, tid, s_magic);
            } else if (blur) {
                if (nh == 1) flex_wpass<1>(s_xs + k0 * strip_w, rh, quads, strip_w, s_xw, s_wq, s_t1, g.rwp, sb, c0, rw, kc * rh, tid, s_magic);
                else flex_wpass<2>(s_xs + k0 * strip_w, rh, quads, strip_w, s_xw, s_wq, s_t1, g.rwp, sb, c0, rw, kc * rh, tid, s_magic);
            } else {
                // the window itself, bit exact: output words (bytes outside the window masked to zero) parked in t1
                const FastDiv fd_nq(g.nq, s_magic), fd_rh(rh, s_magic);
                const uint32_t sh = (uint32_t)(cb - sb) * 8u;
                uint32_t *t1w = reinterpret_cast<uint32_t *>(s_t1);
                const uint32_t *sp0 = s_xs + k0 * strip_w + (c0 >> 2);
                for (int i = tid; i < kc * rh * g.nq; i += kFlexThreads) {
                    const int row = fd_nq.div(i), q = i - row * g.nq;
                    const int kk = fd_rh.div(row), y = row - kk * rh;
                    const uint32_t *sp = sp0 + kk * strip_w + y * quads + q;
                    uint32_t word = __funnelshift_r(sp[0], sp[1], sh);
                    if (q == 0) word &= g.m_first;
                    if (q == g.nq - 1) word &= g.m_last;
                    t1w[i] = word;
                }
            }
            if (last || VARIANT == AGYM_OUT_RESIZE_FOV) cp_async_wait<0>();      // H operator
            __syncthreads();                   // #2: t1 complete; after the last group s_x / s_wq / s_xw are free
            if (last && boss) {
                fetch_strips((j + 1) & (kWin - 1));                    // s_x is free: the next env's windows
                finish_env(pend, (j + 2) & (kWin - 1));                // read by the prefetch after the NEXT env's #2
            }
            if (!worker) continue;
            if (last) prefetch((j + 1) & (kWin - 1));
            if (VARIANT == AGYM_OUT_RESIZE_FOV) {
                glimpse_hpass(s_t1, rh, s_xh, reinterpret_cast<const float *>(s_wh2), th, reinterpret_cast<uint8_t *>(s_tile) + k0 * oh * ow,
                              oh, ow, kc, tid, s_magic);
            } else if (blur) {
                switch (th) {
                    case 3: flex_hpass<3, kPeriph>(g, s_t1, s_wh2, s_xh, s_tile, k0, kc, th, tid, s_magic); break;
                    case 4: flex_hpass<4, kPeriph>(g, s_t1, s_wh2, s_xh, s_tile, k0, kc, th, tid, s_magic); break;
                    case 5: flex_hpass<5, kPeriph>(g, s_t1, s_wh2, s_xh, s_tile, k0, kc, th, tid, s_magic); break;
                    case 6: flex_hpass<6, kPeriph>(g, s_t1, s_wh2, s_xh, s_tile, k0, kc, th, tid, s_magic); break;
                    default: flex_hpass<0, kPeriph>(g, s_t1, s_wh2, s_xh, s_tile, k0, kc, th, tid, s_magic); break;
                }
            } else {
                const FastDiv fd_nq(g.nq, s_magic), fd_rh(rh, s_magic);
                const uint32_t *t1w = reinterpret_cast<const uint32_t *>(s_t1);
                for (int i = tid; i < kc * rh * g.nq; i += kFlexThreads) {
                    const int row = fd_nq.div(i), q = i - row * g.nq;
                    const int kk = fd_rh.div(row), y = row - kk * rh;
                    if (y >= g.vh) continue;
                    uint32_t *d = s_tile + ((k0 + kk) * oh + oy + y) * g.ow4 + g.wlo + q;
                    if (kPeriph) {   // the edge words keep the background's bytes (t1w is zero outside the window)
                        const uint32_t m = (q == 0 ? g.m_first : 0xffffffffu) & (q == g.nq - 1 ? g.m_last : 0xffffffffu);
                        *d = (*d & ~m) | t1w[i];
                    } else {
                        *d = t1w[i];
                    }
                }
            }
        }
        fence_async_smem();
        __syncthreads();                       // #3: tile complete
        const bool words = VARIANT == AGYM_OUT_RESIZE_FOV && word_store;
        if (boss && !words) {
            bulk_s2g(out + (size_t)n * tile_bytes, s_tile, (uint32_t)tile_bytes);
            bulk_commit();
        }
        // uniform: the tile leaves as words, or its normalised copy is written; the tile is next written after barrier #1
        // of the following env, which comes after this in every thread's program order
        if (words) {
            uint32_t *o = reinterpret_cast<uint32_t *>(out + (size_t)n * tile_bytes);
            for (int i = threadIdx.x; i < (tile_bytes >> 2); i += (int)blockDim.x) o[i] = s_tile[i];
        }
        if (p.norm_out) {
            if (VARIANT == AGYM_OUT_RESIZE_FOV && (tile_bytes & 15)) {
                const int nw = tile_bytes >> 2;
                for (int i = threadIdx.x; i < nw; i += (int)blockDim.x) norm_store4(p.norm_dt, s_tile[i], p.norm_out, (size_t)n * nw + i);
            } else {
                const uint4 *t4 = reinterpret_cast<const uint4 *>(s_tile);
                const int nv = tile_bytes >> 4;
                for (int i = threadIdx.x; i < nv; i += (int)blockDim.x) norm_store16(p.norm_dt, t4[i], p.norm_out, (size_t)n * nv + i);
            }
        }
    }
    cp_async_wait<0>();
    if (boss) {
        bulk_wait_read<0>();
    }
}


}  // namespace

// --------------------------------------------------------------------------- launchers
cudaError_t launch_observe_flexible(const DevPlan &p, const uint8_t *ring, const int32_t *head, const float *pcache,
                                    const double *action, const int32_t *atype, const uint8_t *ctrl, int32_t *loc,
                                    int32_t *res, int variant, int pad_h, int pad_w, uint8_t *out, int32_t *err,
                                    void *norm_out, int norm_dt, cudaStream_t st) {
    cudaError_t e;
    DevPlan q = p;
    q.err = err;
    q.norm_out = norm_out; q.norm_dt = norm_dt;
    const size_t out_bytes = (size_t)p.N * p.K *
                             (variant == AGYM_OUT_CROP ? (size_t)pad_h * pad_w : variant == AGYM_OUT_RESIZE_FOV ? (size_t)p.f_h * p.f_w : (size_t)p.plane);
    auto finish = [&](cudaError_t r) {   // kernels without the fused normalised store: a separate pass over the u8 output
        if (r != cudaSuccess || !norm_out) return r;
        if (out_bytes % 16 != 0) return cudaErrorInvalidValue;
        return launch_normalize(out, out_bytes, norm_dt, norm_out, st);
    };
    const bool glimpse = variant == AGYM_OUT_RESIZE_FOV, periph = variant == kOutPeriph;
    // the peripheral variant's squeeze arrives by one bulk copy per env and is expanded by the two-tap tables
    const size_t sq_bytes = periph ? 4 * (size_t)p.K * p.p_h * p.p_w : 0;
    const bool periph_ok = !periph || (p.fast_expand && sq_bytes % 16 == 0 && (reinterpret_cast<uintptr_t>(pcache) & 15) == 0);
    if (variant != AGYM_OUT_RESIZE_FULL && p.flexb && p.flexq && periph_ok && !g_disable_std && !g_flex_old) {
        // persistent kernel, 2 CTAs per SM: whatever the fixed buffers leave of ~113 KB goes to t1
        const int oh = variant == AGYM_OUT_CROP ? pad_h : glimpse ? p.f_h : p.S_h;
        const int ow = variant == AGYM_OUT_CROP ? pad_w : glimpse ? p.f_w : p.S_w;
        const size_t tile = (size_t)p.K * oh * ow;
        const size_t fixed = a16(a16(a16(tile) + 4 * (size_t)p.K * p.S_h * (p.S_w / 4 + 2)) + sq_bytes) +
                             4 * ((size_t)p.S_w * 8 + 2 * (size_t)p.S_h * p.blur_tmax + p.S_w + p.S_h) + 16;
        // floats: one / all K frames of the largest window (the glimpse keeps f_w columns of each window row)
        const size_t one = (size_t)p.S_h * (glimpse ? p.f_w : p.S_w + 4), all = (size_t)p.K * one;
        // + static shared memory + 1 KB reserved per CTA: two CTAs per SM (233,472 B).  RGB plans whose fixed buffers do
        // not leave one window's t1 in that budget (mask_out at 3 frames x 3 planes: 133 KB of tile and strips; the
        // peripheral variant adds 14,400 B of squeeze) run one CTA per SM with the whole SM's shared memory instead
        const int ctas_per_sm = (p.C == 3 && fixed + 4 * one > 114000) ? 1 : 2;
        const size_t budget = ctas_per_sm == 2 ? 114000 : 225000;
        const size_t room = budget > fixed ? ((budget - fixed) / 4) & ~size_t(3) : 0;
        const size_t t1_cap = std::min(all, room);
        // the glimpse's tile leaves by the bulk store when it can, as 4-byte words otherwise; its fp32 operators take the
        // places of the fixed-point W operator (S_w * 8 words) and the duplicated H operator (2 * S_h * blur_tmax words)
        const bool bulk_out = tile % 16 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
        const bool out_ok = glimpse ? tile % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0 &&
                                          (size_t)p.f_w * p.fov_tmax <= (size_t)p.S_w * 8 &&
                                          (size_t)p.f_h * p.fov_tmax <= 2 * (size_t)p.S_h * p.blur_tmax
                                    : bulk_out && ow % 4 == 0 && (size_t)p.K * p.f_h * (p.S_w / 4 + 1) <= t1_cap;
        if (out_ok && t1_cap >= one &&
            p.plane % 16 == 0 && p.S_w % 4 == 0 && (reinterpret_cast<uintptr_t>(ring) & 15) == 0) {   // strip copies
            const size_t fs = fixed + 4 * t1_cap;
            int dev = 0, sms = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            const int grid = std::min(p.N, ctas_per_sm * sms);
            // the env-claim counter starts every launch at zero (stream-ordered; a launch that faulted cannot leave it armed)
            if ((e = cudaMemsetAsync(p.flex_counters, 0, 16, st)) != cudaSuccess) return e;
            if (variant == AGYM_OUT_CROP) {
                if ((e = set_smem(k_observe_flexible_v3<AGYM_OUT_CROP>, fs)) != cudaSuccess) return e;
                k_observe_flexible_v3<AGYM_OUT_CROP><<<grid, kFlexThreads + 32, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, (int)t1_cap, out, p.flex_counters, 0, nullptr);
            } else if (periph) {
                if ((e = set_smem(k_observe_flexible_v3<kOutPeriph>, fs)) != cudaSuccess) return e;
                k_observe_flexible_v3<kOutPeriph><<<grid, kFlexThreads + 32, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, (int)t1_cap, out, p.flex_counters, 0, pcache);
            } else if (glimpse) {
                if ((e = set_smem(k_observe_flexible_v3<AGYM_OUT_RESIZE_FOV>, fs)) != cudaSuccess) return e;
                k_observe_flexible_v3<AGYM_OUT_RESIZE_FOV><<<grid, kFlexThreads + 32, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, (int)t1_cap, out, p.flex_counters, bulk_out ? 0 : 1, nullptr);
            } else {
                if ((e = set_smem(k_observe_flexible_v3<AGYM_OUT_MASK>, fs)) != cudaSuccess) return e;
                k_observe_flexible_v3<AGYM_OUT_MASK><<<grid, kFlexThreads + 32, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, (int)t1_cap, out, p.flex_counters, 0, nullptr);
            }
            return cudaGetLastError();
        }
    }
    if ((variant == AGYM_OUT_CROP || variant == AGYM_OUT_MASK) && p.flexb && !g_disable_std) {
        const int oh = variant == AGYM_OUT_CROP ? pad_h : p.S_h, ow = variant == AGYM_OUT_CROP ? pad_w : p.S_w;
        const size_t tile = (size_t)p.K * oh * ow;
        // t1: one padded window of any size (S_h x S_w), or all K frames of windows up to ~50 x 52
        const int t1_cap = std::max(p.S_h * ((p.S_w + 3) & ~3), std::min(p.K * 50 * 52, p.K * p.S_h * ((p.S_w + 3) & ~3)));
        const size_t fs = tile + 4 * ((size_t)p.K * p.S_h * (p.S_w / 4 + 1) + (size_t)t1_cap +
                                      (size_t)(p.S_w + p.S_h) * p.blur_tmax + p.S_w + p.S_h);
        if (tile % 16 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && fs <= 200 * 1024) {
            if (variant == AGYM_OUT_CROP) {
                if ((e = set_smem(k_observe_flexible_fast<AGYM_OUT_CROP>, fs)) != cudaSuccess) return e;
                k_observe_flexible_fast<AGYM_OUT_CROP><<<p.N, kThreads, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, t1_cap, out);
            } else {
                if ((e = set_smem(k_observe_flexible_fast<AGYM_OUT_MASK>, fs)) != cudaSuccess) return e;
                k_observe_flexible_fast<AGYM_OUT_MASK><<<p.N, kThreads, fs, st>>>(q, ring, head, action, atype, ctrl, loc, res, oh, ow, t1_cap, out);
            }
            return finish(cudaGetLastError());
        }
    }
    // window buffers; the peripheral variant adds the background plane and, for generic expand tables, squeeze + W pass
    const size_t smem = sizeof(float) * 2 * (size_t)p.plane +
                        (periph ? p.plane + sizeof(float) * ((size_t)p.p_h * p.p_w + (size_t)p.p_h * p.S_w) : 0);
#define AGYM_LAUNCH_FLEX(V)                                                                              \
    if ((e = set_smem(k_observe_flexible<V>, smem)) != cudaSuccess) return e;                            \
    k_observe_flexible<V><<<p.N, kThreads, smem, st>>>(q, ring, head, action, atype, ctrl, loc, res, pad_h, pad_w, out, pcache);
    if (periph) { AGYM_LAUNCH_FLEX(kOutPeriph) }
    else if (variant == AGYM_OUT_CROP) { AGYM_LAUNCH_FLEX(AGYM_OUT_CROP) }
    else if (variant == AGYM_OUT_MASK) { AGYM_LAUNCH_FLEX(AGYM_OUT_MASK) }
    else if (glimpse) { AGYM_LAUNCH_FLEX(AGYM_OUT_RESIZE_FOV) }
    else { AGYM_LAUNCH_FLEX(AGYM_OUT_RESIZE_FULL) }
#undef AGYM_LAUNCH_FLEX
    return finish(cudaGetLastError());
}


}  // namespace agym
