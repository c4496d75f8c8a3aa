// sm_100a kernels: ingest (raw simulator frames -> frame-stack ring) and stack.
#include "agym_device.cuh"

namespace agym {

namespace {

// ------------------------------------------------------------------------ ingest: Atari
// AtariEnv._get_state + the frame logic of _step/_reset (atari_env.py:73-75, 80-82, 91,
// 111-114, 121-133): gray -> cv2.resize(INTER_LINEAR) for frame A and frame B separately,
// max of the two resized frames, push.  Shared memory holds, per frame, only the two source
// rows every output row samples (raw rows the resize never reads are not fetched).
template <int CH>
__global__ void __launch_bounds__(kThreads) k_ingest_atari(const __grid_constant__ DevPlan p,
                                                           const uint8_t *__restrict__ fa,
                                                           const uint8_t *__restrict__ fb,
                                                           const uint8_t *__restrict__ flags, uint8_t *__restrict__ ring,
                                                           int32_t *__restrict__ head, float *__restrict__ pcache) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int n = blockIdx.x, tid = threadIdx.x;
    const int fl = flags[n];
    if (fl & AGYM_FLAG_IDLE) return;
    const int slot = (head[n] + 1) % p.K;

    int32_t *t_xs0 = reinterpret_cast<int32_t *>(smem);
    int32_t *t_xs1 = t_xs0 + p.S_w, *t_xcf = t_xs1 + p.S_w;
    int32_t *t_ys0 = t_xcf + p.S_w, *t_ys1 = t_ys0 + p.S_h, *t_ycf = t_ys1 + p.S_h;
    uint8_t *s_gray = smem + align16(sizeof(int32_t) * 3 * (p.S_w + p.S_h));
    const int rows2 = 2 * p.S_h;                       // staged rows per frame
    const size_t gray_bytes = (size_t)rows2 * p.raw_w; // per frame
    uint8_t *s_frame = s_gray + align16(2 * gray_bytes);
    float *s_t1 = reinterpret_cast<float *>(s_frame + align16(p.plane));

    for (int i = tid; i < p.S_w; i += kThreads) {
        t_xs0[i] = p.cx_s0[i]; t_xs1[i] = p.cx_s1[i]; t_xcf[i] = p.cx_coef[i];
    }
    for (int i = tid; i < p.S_h; i += kThreads) {
        t_ys0[i] = p.cy_s0[i]; t_ys1[i] = p.cy_s1[i]; t_ycf[i] = p.cy_coef[i];
    }
    __syncthreads();  // also orders every thread's read of head[n] before the update below
    if (tid == 0) head[n] = slot;

    // ---- stage: gray rows of the valid frames -> shared memory
    const int vpr = p.raw_w / 16;  // 16-pixel groups per row
    const FastDiv fd_vpr(vpr);
    const size_t frame_bytes = (size_t)p.raw_h * p.raw_w * CH;
#pragma unroll 1
    for (int fr = 0; fr < 2; ++fr) {
        if (!(fl & (1 << fr))) continue;
        const uint8_t *src = (fr ? fb : fa) + frame_bytes * n;
        uint8_t *dst = s_gray + gray_bytes * fr;
#pragma unroll 2
        for (int t = tid; t < rows2 * vpr; t += kThreads) {
            const int sr = fd_vpr.div(t), g = t - sr * vpr;
            const int srow = (sr & 1) ? t_ys1[sr >> 1] : t_ys0[sr >> 1];
            uint4 o;
            if (CH == 1) {
                o = ld_stream128(src + (size_t)srow * p.raw_w + 16 * g);
            } else {
                const uint8_t *q = src + ((size_t)srow * p.raw_w + 16 * g) * 3;
                uint32_t w[12];
                *reinterpret_cast<uint4 *>(w) = ld_stream128(q);
                *reinterpret_cast<uint4 *>(w + 4) = ld_stream128(q + 16);
                *reinterpret_cast<uint4 *>(w + 8) = ld_stream128(q + 32);
                o = luma16(w, (2u * p.lw0) | ((2u * p.lw1) << 16), 2u * p.lw2);
            }
            *reinterpret_cast<uint4 *>(dst + (size_t)sr * p.raw_w + 16 * g) = o;
        }
    }
    // hard reset: the other K-1 slots (and their cache entries) become zero frames
    if (fl & AGYM_FLAG_HARD_RESET) {
        const int words = p.plane / 4;
        for (int k = 0; k < p.K; ++k) {
            if (k == slot) continue;
            uint32_t *z = reinterpret_cast<uint32_t *>(ring + ((size_t)n * p.K + k) * p.plane);
            for (int i = tid; i < words; i += kThreads) z[i] = 0u;
            if (pcache) {
                float *zc = pcache + ((size_t)n * p.K + k) * p.p_h * p.p_w;
                for (int i = tid; i < p.p_h * p.p_w; i += kThreads) zc[i] = 0.f;
            }
        }
    }
    __syncthreads();

    // ---- resize both frames (11-bit fixed point, horizontal then vertical), max, store
    const int wpr = p.S_w / 4;  // output words per row
    const FastDiv fd_wpr(wpr);
    uint32_t *out_words = reinterpret_cast<uint32_t *>(ring + ((size_t)n * p.K + slot) * p.plane);
    uint32_t *frame_words = reinterpret_cast<uint32_t *>(s_frame);
    for (int t = tid; t < p.plane / 4; t += kThreads) {
        const int y = fd_wpr.div(t), q = t - y * wpr;
        const int ycf = t_ycf[y];
        const int b0 = ycf & 0xffff, b1 = ycf >> 16;
        uint32_t word = 0u;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int x = 4 * q + i;
            const int s0 = t_xs0[x], s1 = t_xs1[x], xcf = t_xcf[x];
            const int c0 = xcf & 0xffff, c1 = xcf >> 16;
            int m = 0;
#pragma unroll
            for (int fr = 0; fr < 2; ++fr) {
                if (!(fl & (1 << fr))) continue;
                const uint8_t *r0 = s_gray + gray_bytes * fr + (size_t)(2 * y) * p.raw_w;
                const uint8_t *r1 = r0 + p.raw_w;
                const int h0 = r0[s0] * c0 + r0[s1] * c1;
                const int h1 = r1[s0] * c0 + r1[s1] * c1;
                const int v = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
                m = max(m, v);
            }
            word |= (uint32_t)min(m, 255) << (8 * i);
        }
        out_words[t] = word;
        if (pcache) frame_words[t] = word;
    }
    if (pcache) {  // uniform branch
        __syncthreads();
        squeeze_to_cache(p, s_frame, s_t1, pcache + ((size_t)n * p.K + slot) * p.p_h * p.p_w, tid, kThreads);
    }
}

// Squeeze along W straight from a u8 frame in shared memory (fov_env.py:367, W pass): every
// output column reads one 16-byte window, realigned with funnel shifts so that the byte ->
// float conversions use compile-time byte selectors (I2F.U8 Rx.Bn).
__device__ __forceinline__ void squeeze_w_fast(const DevPlan &p, const uint8_t *s_frame, float *s_t1, int tid, int nt) {
    const int total = p.S_h * p.p_w;
    const FastDiv fd(p.p_w);
    const int nq = p.sqw_taps4 >> 2;
    for (int t = tid; t < total; t += nt) {
        const int y = fd.div(t), i = t - y * p.p_w;
        const int2 o = __ldg(p.sqw_ofs + i);
        const uint32_t *src = reinterpret_cast<const uint32_t *>(s_frame + y * p.S_w + o.x);
        const uint32_t w0 = src[0], w1 = src[1], w2 = src[2], w3 = src[3];
        const uint32_t a[4] = {__funnelshift_r(w0, w1, o.y), __funnelshift_r(w1, w2, o.y), __funnelshift_r(w2, w3, o.y),
                               w3 >> o.y};
        const float4 *wt = reinterpret_cast<const float4 *>(p.sqw_w + i * p.sqw_taps4);
        float acc = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (q < nq) {
                const float4 w = __ldg(wt + q);
                const uint32_t v = a[q];
                acc = fmaf(w.x, (float)(v & 0xffu), acc);
                acc = fmaf(w.y, (float)((v >> 8) & 0xffu), acc);
                acc = fmaf(w.z, (float)((v >> 16) & 0xffu), acc);
                acc = fmaf(w.w, (float)(v >> 24), acc);
            }
        }
        s_t1[t] = acc;
    }
}

// Fast ingest (geometry checked at plan creation): the horizontal pass as IDP.2A on byte pairs
// picked with PRMT from two aligned words, the vertical pass as two IMAD.HI; one thread owns
// two adjacent output columns and walks a segment of output rows.
template <int CH>
__global__ void __launch_bounds__(kThreads) k_ingest_atari_fast(const __grid_constant__ DevPlan p,
                                                                const uint8_t *__restrict__ fa,
                                                                const uint8_t *__restrict__ fb,
                                                                const uint8_t *__restrict__ flags,
                                                                uint8_t *__restrict__ ring, int32_t *__restrict__ head,
                                                                float *__restrict__ pcache) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int n = blockIdx.x, tid = threadIdx.x;
    const int fl = flags[n];
    if (fl & AGYM_FLAG_IDLE) return;
    const int slot = (head[n] + 1) % p.K;
    const int rows2 = 2 * p.S_h;
    const size_t gray_bytes = (size_t)rows2 * p.raw_w;
    // one frame's sampled rows at a time: half the shared memory, twice the CTAs per SM to hide the
    // latency of the global loads (this kernel has no prefetch pipeline)
    uint8_t *s_gray = smem;
    uint8_t *s_frame = s_gray + align16(gray_bytes + 16);
    float *s_t1 = reinterpret_cast<float *>(s_frame + align16(p.plane + 16));
    __syncthreads();  // every thread has read head[n]
    if (tid == 0) head[n] = slot;

    if (fl & AGYM_FLAG_HARD_RESET) {
        const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
        for (int k = 0; k < p.K; ++k) {
            if (k == slot) continue;
            uint4 *z = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + k) * p.plane);
            for (int i = tid; i < p.plane / 16; i += kThreads) z[i] = z4;
            if (pcache) {
                float *zc = pcache + ((size_t)n * p.K + k) * p.p_h * p.p_w;
                for (int i = tid; i < p.p_h * p.p_w; i += kThreads) zc[i] = 0.f;
            }
        }
    }
    if (!(fl & 3))  // no frame at all (game over before t == 2): a zero frame (atari_env.py:121,132)
        for (int i = tid; i < p.plane / 16; i += kThreads) reinterpret_cast<uint4 *>(s_frame)[i] = make_uint4(0u, 0u, 0u, 0u);

    const int vpr = p.raw_w / 16;
    const FastDiv fd_vpr(vpr);
    const size_t frame_bytes = (size_t)p.raw_h * p.raw_w * CH;
    const int pairs = p.S_w >> 1, segs = kThreads / pairs;
    const int g = tid / pairs, pi = tid - g * pairs;
    const int4 px = g < segs ? __ldg(p.cx_pair + pi) : make_int4(0, 0, 0, 0);  // {aligned byte offset, PRMT selector, coef(x0), coef(x0+1)}
    const int rows_per = (p.S_h + segs - 1) / segs;
    const int y_begin = g * rows_per, y_end = g < segs ? min(p.S_h, (g + 1) * rows_per) : y_begin;
    bool first = true;
#pragma unroll 1
    for (int fr = 0; fr < 2; ++fr) {
        if (!(fl & (1 << fr))) continue;
        const uint8_t *src = (fr ? fb : fa) + frame_bytes * n;
#pragma unroll 4
        for (int t = tid; t < rows2 * vpr; t += kThreads) {
            const int sr = fd_vpr.div(t), gg = t - sr * vpr;
            const int srow = __ldg(((sr & 1) ? p.cy_s1 : p.cy_s0) + (sr >> 1));
            uint4 o;
            if (CH == 1) {
                o = ld_stream128(src + (size_t)srow * p.raw_w + 16 * gg);
            } else {
                const uint8_t *q = src + ((size_t)srow * p.raw_w + 16 * gg) * 3;
                uint32_t w[12];
                *reinterpret_cast<uint4 *>(w) = ld_stream128(q);
                *reinterpret_cast<uint4 *>(w + 4) = ld_stream128(q + 16);
                *reinterpret_cast<uint4 *>(w + 8) = ld_stream128(q + 32);
                o = luma16(w, (2u * p.lw0) | ((2u * p.lw1) << 16), 2u * p.lw2);
            }
            *reinterpret_cast<uint4 *>(s_gray + (size_t)sr * p.raw_w + 16 * gg) = o;
        }
        __syncthreads();
        for (int y = y_begin; y < y_end; ++y) {
            const int2 bs = __ldg(p.cy_bs + y);  // {b0 << 16, b1 << 16}
            const uint8_t *r0 = s_gray + (size_t)(2 * y) * p.raw_w + px.x;
            const uint32_t a0 = *reinterpret_cast<const uint32_t *>(r0);
            const uint32_t a1 = *reinterpret_cast<const uint32_t *>(r0 + 4);
            const uint32_t b0 = *reinterpret_cast<const uint32_t *>(r0 + p.raw_w);
            const uint32_t b1 = *reinterpret_cast<const uint32_t *>(r0 + p.raw_w + 4);
            const uint32_t qa = __byte_perm(a0, a1, (uint32_t)px.y), qb = __byte_perm(b0, b1, (uint32_t)px.y);
            const uint32_t h00 = __dp2a_lo((uint32_t)px.z, qa, 0u), h01 = __dp2a_hi((uint32_t)px.w, qa, 0u);
            const uint32_t h10 = __dp2a_lo((uint32_t)px.z, qb, 0u), h11 = __dp2a_hi((uint32_t)px.w, qb, 0u);
            // never above 255: b0 + b1 = 2048 and h >> 4 <= 32640
            uint32_t v0 = (__umulhi((uint32_t)bs.x, h00 >> 4) + __umulhi((uint32_t)bs.y, h10 >> 4) + 2u) >> 2;
            uint32_t v1 = (__umulhi((uint32_t)bs.x, h01 >> 4) + __umulhi((uint32_t)bs.y, h11 >> 4) + 2u) >> 2;
            uint16_t *o = reinterpret_cast<uint16_t *>(s_frame + y * p.S_w + 2 * pi);
            if (!first) {  // max with the other frame's resized pixel (atari_env.py:132)
                const uint32_t prev = *o;
                v0 = max(v0, prev & 0xffu);
                v1 = max(v1, prev >> 8);
            }
            *o = (uint16_t)(v0 | (v1 << 8));
        }
        first = false;
        __syncthreads();
    }
    uint4 *out4 = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + slot) * p.plane);
    for (int i = tid; i < p.plane / 16; i += kThreads) out4[i] = reinterpret_cast<const uint4 *>(s_frame)[i];
    if (pcache) {  // uniform
        float *dst = pcache + ((size_t)n * p.K + slot) * p.p_h * p.p_w;
        if (p.fast_squeeze) squeeze_w_fast(p, s_frame, s_t1, tid, kThreads);
        else resample_w<uint8_t>(s_frame, p.S_w, s_t1, p.p_w, p.S_h, p.sq_w, tid, kThreads);
        __syncthreads();
        resample_h<float>(s_t1, p.p_w, dst, p.p_w, p.p_w, p.sq_h, tid, kThreads);
    }
}


// Persistent, TMA-fed ingest for gray frames.  Every CTA walks the env batch in "units" of R
// output rows; for each unit ONE cp.async.bulk per frame brings the contiguous span of source
// rows the unit samples into a ring of shared-memory stages, tracked by full/empty mbarriers
// (the canonical TMA producer/consumer pipeline): warp 8 is the producer, warps 0-7 resize.
// HBM streaming and the fixed-point arithmetic therefore overlap inside every CTA.
// RAW_W / S_W > 0 bake the strides of the standard geometry (210x160 -> 84x84) into the
// instruction immediates; 0 = take them from the plan.
constexpr int kIngestThreads = kThreads + 32;

// TM: the standard 2.5x vertical scale samples raw rows {5m, 5m+1} (even output rows) and {5m+3, 5m+4} (odd ones)
// and never row 5m+2.  The frames are then viewed as a 4-D tensor [env][period of 5 rows][row in period][row bytes]
// and a unit's rows arrive as TWO tiled tensor copies per frame (boxes of 2 rows x R/2 periods at row 0 and at
// row 3 of the period): the unsampled fifth of every frame never leaves HBM, with as few copies as before.
template <int RAW_W, int S_W, int CH, bool TM, int NS>  // RAW_W: BYTES per raw row (pixels * CH) when baked in; NS: stages
__global__ void __launch_bounds__(kIngestThreads, 3) k_ingest_atari_tma(const __grid_constant__ DevPlan p,
                                                                        const uint8_t *__restrict__ fa,
                                                                        const uint8_t *__restrict__ fb,
                                                                        const uint8_t *__restrict__ flags,
                                                                        uint8_t *__restrict__ ring,
                                                                        int32_t *__restrict__ head,
                                                                        float *__restrict__ pcache, int units,
                                                                        int span_rows,
                                                                        const __grid_constant__ CUtensorMap tma,
                                                                        const __grid_constant__ CUtensorMap tmb) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint8_t *smem = smem_raw + (TM ? ((128u - (smem_u32(smem_raw) & 127u)) & 127u) : 0u);   // tensor copies land on 128-byte lines
    __shared__ __align__(8) uint64_t full[NS], empty[NS];
    constexpr int kEnvWin = 64;
    __shared__ int s_envfl[kEnvWin], s_envhd[kEnvWin];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int N = p.N, K = p.K;
    const int raw_w = RAW_W ? RAW_W : p.raw_w * CH;               // bytes per raw row
    const int S_w = S_W ? S_W : p.S_w;
    const int R = p.S_h / units;                          // output rows per unit
    const int box_bytes = R * raw_w;                      // TM: the R/2 x 2 rows of one tensor copy ...
    const int block_bytes = (box_bytes + 127) & ~127;     // ... which must land on a 128-byte line
    const int frame_stride = TM ? 2 * block_bytes + 128 : span_rows * raw_w + 16;  // one frame's staged rows of a unit (+ pad)
    const int stage_bytes = (2 * frame_stride + 15) & ~15;
    uint8_t *stages = smem;
    uint8_t *s_frame = stages + NS * stage_bytes;
    float *s_t1 = reinterpret_cast<float *>(s_frame + align16(p.plane + 16));
    int4 *s_row = reinterpret_cast<int4 *>(s_t1 + (pcache ? p.S_h * p.p_w : 0));  // [S_h] {ofs0, ofs1, b0<<16, b1<<16}
    int2 *s_span = reinterpret_cast<int2 *>(s_row + p.S_h);                       // [units] {first row, bytes}
    float *s_sqw = reinterpret_cast<float *>(s_span + ((units + 1) & ~1));        // [p_w][taps4], 16-byte aligned
    uint32_t *s_sqq = reinterpret_cast<uint32_t *>(s_sqw + (pcache ? p.p_w * 16 : 0));  // [p_w][8] fixed-point W weights
    float *s_sqh = reinterpret_cast<float *>(s_sqq + (pcache ? p.p_w * 8 : 0));         // [p_h][taps] H-pass weights
    int32_t *s_sqx = reinterpret_cast<int32_t *>(s_sqh + (pcache ? p.p_h * p.sq_h.taps : 0));  // [p_h] first source row
    const size_t frame_bytes = (size_t)p.raw_h * raw_w;

    pdl_launch_dependents();
    if (tid == 0) {
        for (int i = 0; i < NS; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], kThreads / 32); }
        mbar_fence_init();
    }
    for (int y = tid; y < p.S_h; y += kIngestThreads) {
        const int2 bs = __ldg(p.cy_bs + y);
        if (TM) {   // even rows of the unit in the first block, odd rows in the second, two staged rows each
            const int yy = y - (y / R) * R;
            const int o = ((yy & 1) ? block_bytes : 0) + (yy >> 1) * 2 * raw_w;
            s_row[y] = make_int4(o, o + raw_w, bs.x, bs.y);
        } else {
            const int lo = __ldg(p.cy_s0 + (y / R) * R);     // first source row of this row's unit
            s_row[y] = make_int4((__ldg(p.cy_s0 + y) - lo) * raw_w, (__ldg(p.cy_s1 + y) - lo) * raw_w, bs.x, bs.y);
        }
    }
    for (int u = tid; u < units; u += kIngestThreads) {
        const int lo = __ldg(p.cy_s0 + u * R), hi = __ldg(p.cy_s1 + u * R + R - 1);
        s_span[u] = make_int2(lo, (hi - lo + 1) * raw_w);
    }
    if (pcache && p.fast_squeeze)
        for (int i = tid; i < p.p_w * p.sqw_taps4; i += kIngestThreads) s_sqw[i] = __ldg(p.sqw_w + i);
    if (pcache) {
        for (int i = tid; i < p.p_w * 8; i += kIngestThreads) s_sqq[i] = p.squeeze_q ? __ldg(p.sqw_q + i) : 0u;
        for (int i = tid; i < p.p_h * p.sq_h.taps; i += kIngestThreads) s_sqh[i] = __ldg(p.sq_h.w + i);
        for (int i = tid; i < p.p_h; i += kIngestThreads) s_sqx[i] = __ldg(p.sq_h.xmin + i);
    }
    __syncthreads();
    pdl_wait();   // frames, flags, ring, head, pcache: not before the previous kernel in the stream has finished

    // unit `it` of this CTA: env = blockIdx.x + (it / units) * gridDim.x, part = it % units
    const int my_envs = (N - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
    const int my_units = my_envs * units;

    if (warp == kThreads / 32) {
        // ------------------------------------------------------------------ producer warp
        if (lane == 0) {
            int n = blockIdx.x, part = 0, st = 0, ph = 1;  // ph: parity of the empty-barrier phase to wait for
            for (int it = 0; it < my_units; ++it) {
                if (it >= NS) mbar_wait<true>(&empty[st], ph);
                const int fl = flags[n];
                const int2 span = s_span[part];
                const int nvalid = (fl & AGYM_FLAG_IDLE) ? 0 : __popc(fl & 3);
                uint8_t *dst = stages + st * stage_bytes;
                if (TM) {
                    mbar_expect_tx(&full[st], (uint32_t)(nvalid * 2 * box_bytes));
                    const int m0 = (R >> 1) * part;
                    if (nvalid && (fl & AGYM_FLAG_FRAME_A)) {
                        tensor_g2s_4d(dst, &tma, &full[st], 0, 0, m0, n);
                        tensor_g2s_4d(dst + block_bytes, &tma, &full[st], 0, 3, m0, n);
                    }
                    if (nvalid && (fl & AGYM_FLAG_FRAME_B)) {
                        tensor_g2s_4d(dst + frame_stride, &tmb, &full[st], 0, 0, m0, n);
                        tensor_g2s_4d(dst + frame_stride + block_bytes, &tmb, &full[st], 0, 3, m0, n);
                    }
                } else {
                    mbar_expect_tx(&full[st], (uint32_t)(nvalid * span.y));
                    if (nvalid) {
                        const size_t off = frame_bytes * n + (size_t)span.x * raw_w;
                        if (fl & AGYM_FLAG_FRAME_A) bulk_g2s(dst, fa + off, span.y, &full[st]);
                        if (fl & AGYM_FLAG_FRAME_B) bulk_g2s(dst + frame_stride, fb + off, span.y, &full[st]);
                    }
                }
                if (++part == units) { part = 0; n += gridDim.x; }
                if (++st == NS) { st = 0; ph ^= 1; }
            }
        }
        return;
    }

    // ---------------------------------------------------------------------- consumer warps
    const int pairs = S_w >> 1, segs = kThreads / pairs;
    const int g = tid / pairs, pi = tid - g * pairs;
    const bool worker = g < segs;
    const int4 px = worker ? __ldg(p.cx_pair + pi) : make_int4(0, 0, 0, 0);
    // RGB: the four source pixels of this column pair lie among s0 .. s0 + 3 (checked when the plan was made):
    // 12 bytes starting at byte 3 * s0 of the row
    const int s0px = px.x + (px.y & 7);
    const int tap_off = CH == 1 ? px.x : ((3 * s0px) & ~3);
    const uint32_t rgb_sh = (uint32_t)((3 * s0px) & 3) * 8u;
    uint32_t rgb_sel = 0u;
    if (CH == 3) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int rel = ((px.y >> (4 * k)) & 7) - (px.y & 7);  // 0..3: which of the four lumas
            rgb_sel |= (uint32_t)(rel < 2 ? rel : rel + 2) << (4 * k);
        }
    }
    const uint32_t lw_a = (2u * p.lw0) | ((2u * p.lw1) << 16), lw_b = 2u * p.lw2;
    const uint32_t lw_c = (2u * p.lw0) << 16, lw_d = (2u * p.lw1) | ((2u * p.lw2) << 16);
    // the 4 source bytes {s0(x0), s1(x0), s0(x0+1), s1(x0+1)} of one raw row, as the IDP.2A operand
    auto tap4 = [&](const uint8_t *row) -> uint32_t {
        const uint32_t *w = reinterpret_cast<const uint32_t *>(row);
        if (CH == 1) return __byte_perm(w[0], w[1], (uint32_t)px.y);
        // cv2 luma Y = (lw . c + 16384) >> 15 = byte 2 of 2 (lw . c) + 32768, for 4 consecutive RGB pixels:
        // v0 = R0 G0 B0 R1, v1 = G1 B1 R2 G2, v2 = B2 R3 G3 B3
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
        const uint32_t v0 = __funnelshift_r(w0, w1, rgb_sh), v1 = __funnelshift_r(w1, w2, rgb_sh), v2 = __funnelshift_r(w2, w3, rgb_sh);
        const uint32_t y0 = __dp2a_hi(lw_b, v0, __dp2a_lo(lw_a, v0, 32768u));
        const uint32_t y1 = __dp2a_lo(lw_d, v1, __dp2a_hi(lw_c, v0, 32768u));
        const uint32_t y2 = __dp2a_lo(lw_b, v2, __dp2a_hi(lw_a, v1, 32768u));
        const uint32_t y3 = __dp2a_hi(lw_d, v2, __dp2a_lo(lw_c, v2, 32768u));
        return __byte_perm(__byte_perm(y0, y1, 0x0062), __byte_perm(y2, y3, 0x0062), rgb_sel);
    };
    const int rows_per = (R + segs - 1) / segs;
    const int yy_begin = g * rows_per, yy_end = worker ? min(R, yy_begin + rows_per) : yy_begin;
    // squeeze along W: one thread = one output column i, rows in passes
    const int sq_rows = p.fast_squeeze ? kThreads / p.p_w : 0;
    const int sq_i = sq_rows ? tid % p.p_w : 0, sq_y0 = sq_rows ? tid / p.p_w : 0;
    const bool sq_worker = pcache && sq_rows && sq_y0 < sq_rows;
    const int nq = p.sqw_taps4 >> 2;
    const int2 sq_o = sq_worker ? __ldg(p.sqw_ofs + sq_i) : make_int2(0, 0);
    const float4 *sqw4 = reinterpret_cast<const float4 *>(s_sqw + sq_i * p.sqw_taps4);
    const uint4 *sqq4 = reinterpret_cast<const uint4 *>(s_sqq) + 2 * sq_i;  // fixed-point weights of this column

    int slot = 0, fl = 0;
    for (int it = 0, n = blockIdx.x, part = 0, st = 0, ph = 0, je = 0; it < my_units; ++it) {
        if (part == 0) {
            // flags / head of this CTA's next kEnvWin envs are fetched together into shared memory: a load per
            // env, used at once, left every warp waiting ~a microsecond of DRAM latency per env
            if ((je & (kEnvWin - 1)) == 0) {
                consumer_sync();
                if (tid < kEnvWin && (long long)n + (long long)tid * gridDim.x < N) {
                    s_envfl[tid] = flags[n + tid * gridDim.x];
                    s_envhd[tid] = head[n + tid * gridDim.x];
                }
                consumer_sync();
            }
            fl = s_envfl[je & (kEnvWin - 1)];
            slot = s_envhd[je & (kEnvWin - 1)] + 1;
            slot -= slot >= K ? K : 0;
            ++je;
        }
        const bool idle = fl & AGYM_FLAG_IDLE;
        mbar_wait(&full[st], ph);
        if (!idle && yy_begin < yy_end) {
            const uint8_t *base = stages + st * stage_bytes + tap_off;
            const int4 *rw = s_row + part * R + yy_begin;
            uint8_t *o = s_frame + (part * R + yy_begin) * S_w + 2 * pi;
            if ((fl & 3) == 3) {  // both frames (the steady state)
                auto row_both = [&](const int4 t, uint8_t *dst) {
                    const uint8_t *ra = base + t.x, *rb = base + t.y;
                    // max of the two frames taken before the final (x + 2) >> 2, which is monotone; the
                    // result cannot exceed 255 (b0 + b1 = 2048, h >> 4 <= 32640), so cv2's saturate is a no-op
                    uint32_t m0 = 0u, m1 = 0u;
#pragma unroll
                    for (int fr = 0; fr < 2; ++fr) {
                        const uint32_t qa = tap4(ra + fr * frame_stride), qb = tap4(rb + fr * frame_stride);
                        const uint32_t h00 = __dp2a_lo((uint32_t)px.z, qa, 0u), h01 = __dp2a_hi((uint32_t)px.w, qa, 0u);
                        const uint32_t h10 = __dp2a_lo((uint32_t)px.z, qb, 0u), h11 = __dp2a_hi((uint32_t)px.w, qb, 0u);
                        m0 = max(m0, __umulhi((uint32_t)t.z, h00 >> 4) + __umulhi((uint32_t)t.w, h10 >> 4));
                        m1 = max(m1, __umulhi((uint32_t)t.z, h01 >> 4) + __umulhi((uint32_t)t.w, h11 >> 4));
                    }
                    *reinterpret_cast<uint16_t *>(dst) = (uint16_t)(((m0 + 2u) >> 2) | (((m1 + 2u) >> 2) << 8));
                };
#pragma unroll 2
                for (int yy = yy_begin; yy < yy_end; ++yy, ++rw, o += S_w) row_both(*rw, o);
            } else {  // resets / early game-over: one frame or none
                for (int yy = yy_begin; yy < yy_end; ++yy, ++rw, o += S_w) {
                    const int4 t = *rw;
                    uint32_t m0 = 0u, m1 = 0u;
                    for (int fr = 0; fr < 2; ++fr) {
                        if (!(fl & (1 << fr))) continue;
                        const uint8_t *ra = base + t.x + fr * frame_stride, *rb = base + t.y + fr * frame_stride;
                        const uint32_t qa = tap4(ra), qb = tap4(rb);
                        const uint32_t h00 = __dp2a_lo((uint32_t)px.z, qa, 0u), h01 = __dp2a_hi((uint32_t)px.w, qa, 0u);
                        const uint32_t h10 = __dp2a_lo((uint32_t)px.z, qb, 0u), h11 = __dp2a_hi((uint32_t)px.w, qb, 0u);
                        m0 = max(m0, (__umulhi((uint32_t)t.z, h00 >> 4) + __umulhi((uint32_t)t.w, h10 >> 4) + 2u) >> 2);
                        m1 = max(m1, (__umulhi((uint32_t)t.z, h01 >> 4) + __umulhi((uint32_t)t.w, h11 >> 4) + 2u) >> 2);
                    }
                    *reinterpret_cast<uint16_t *>(o) = (uint16_t)(min(m0, 255u) | (min(m1, 255u) << 8));
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[st]);  // this warp is done with the stage
        if (++st == NS) { st = 0; ph ^= 1; }
        if (++part < units) continue;
        part = 0;
        const int n_done = n;
        n += gridDim.x;
        if (idle) continue;
        {
            const int n = n_done;
        consumer_sync();  // the whole 84x84 frame is in s_frame
        if (tid == 0) head[n] = slot;
        if (fl & AGYM_FLAG_HARD_RESET) {
            const uint4 z4 = make_uint4(0u, 0u, 0u, 0u);
            for (int k = 0; k < K; ++k) {
                if (k == slot) continue;
                uint4 *z = reinterpret_cast<uint4 *>(ring + ((size_t)n * K + k) * p.plane);
                for (int i = tid; i < p.plane / 16; i += kThreads) z[i] = z4;
                if (pcache) {
                    float *zc = pcache + ((size_t)n * K + k) * p.p_h * p.p_w;
                    for (int i = tid; i < p.p_h * p.p_w; i += kThreads) zc[i] = 0.f;
                }
            }
        }
        uint4 *out4 = reinterpret_cast<uint4 *>(ring + ((size_t)n * K + slot) * p.plane);
        for (int i = tid; i < p.plane / 16; i += kThreads) out4[i] = reinterpret_cast<const uint4 *>(s_frame)[i];
        if (pcache) {  // uniform
            if (sq_rows && p.squeeze_q) {
                // W pass in 16-bit fixed point: 8 IDP.2A over the aligned 16-byte window, exact integer sum
                if (sq_worker) {
                    const uint4 qa = sqq4[0], qb = sqq4[1];  // live only across this loop
                    for (int y = sq_y0; y < p.S_h; y += sq_rows) {
                        const uint32_t *src = reinterpret_cast<const uint32_t *>(s_frame + y * S_w + sq_o.x);
                        uint32_t acc = __dp2a_lo(qa.x, src[0], 0u);
                        acc = __dp2a_hi(qa.y, src[0], acc);
                        acc = __dp2a_lo(qa.z, src[1], acc);
                        acc = __dp2a_hi(qa.w, src[1], acc);
                        acc = __dp2a_lo(qb.x, src[2], acc);
                        acc = __dp2a_hi(qb.y, src[2], acc);
                        acc = __dp2a_lo(qb.z, src[3], acc);
                        acc = __dp2a_hi(qb.w, src[3], acc);
                        s_t1[y * p.p_w + sq_i] = (float)acc * (1.f / 131072.f);
                    }
                }
            } else if (sq_rows) {
                if (sq_worker) {
                    for (int y = sq_y0; y < p.S_h; y += sq_rows) {
                        const uint32_t *src = reinterpret_cast<const uint32_t *>(s_frame + y * S_w + sq_o.x);
                        const uint32_t w0 = src[0], w1 = src[1], w2 = src[2], w3 = src[3];
                        const uint32_t a[4] = {__funnelshift_r(w0, w1, sq_o.y), __funnelshift_r(w1, w2, sq_o.y),
                                               __funnelshift_r(w2, w3, sq_o.y), w3 >> sq_o.y};
                        float acc = 0.f;
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            if (q < nq) {
                                const uint32_t v = a[q];
                                const float4 w = sqw4[q];
                                acc = fmaf(w.x, (float)(v & 0xffu), acc);
                                acc = fmaf(w.y, (float)((v >> 8) & 0xffu), acc);
                                acc = fmaf(w.z, (float)((v >> 16) & 0xffu), acc);
                                acc = fmaf(w.w, (float)(v >> 24), acc);
                            }
                        }
                        s_t1[y * p.p_w + sq_i] = acc;
                    }
                }
            } else {
                resample_w<uint8_t>(s_frame, S_w, s_t1, p.p_w, p.S_h, p.sq_w, tid, kThreads);
            }
            consumer_sync();
            {   // H pass: out[i][j] = sum_t wh[i][t] * t1[xmin[i] + t][j], weights from shared memory
                float *dst = pcache + ((size_t)n * K + slot) * p.p_h * p.p_w;
                const int pw = p.p_w, taps = p.sq_h.taps, total = p.p_h * pw;
                auto one = [&](int o, int i, int j) {
                    const float *w = s_sqh + i * taps;
                    const float *t = s_t1 + s_sqx[i] * pw + j;
                    float acc0 = 0.f, acc1 = 0.f;
                    int tt = 0;
                    for (; tt + 1 < taps; tt += 2) {
                        acc0 = fmaf(w[tt], t[tt * pw], acc0);
                        acc1 = fmaf(w[tt + 1], t[(tt + 1) * pw], acc1);
                    }
                    if (tt < taps) acc0 = fmaf(w[tt], t[tt * pw], acc0);
                    dst[o] = acc0 + acc1;
                };
                if ((pw & 3) == 0) {
                    // four adjacent columns per thread: one LDS.128 of t1 and one weight per tap serve 4 FFMA
                    const int nq = pw >> 2;
                    const FastDiv fd_nq(nq);
                    for (int o = tid; o < p.p_h * nq; o += kThreads) {
                        const int i = fd_nq.div(o), j = 4 * (o - i * nq);
                        const float *w = s_sqh + i * taps;
                        const float *t = s_t1 + s_sqx[i] * pw + j;
                        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                        for (int tt = 0; tt < taps; ++tt) {
                            const float4 v = *reinterpret_cast<const float4 *>(t + tt * pw);
                            const float wt = w[tt];
                            acc.x = fmaf(wt, v.x, acc.x); acc.y = fmaf(wt, v.y, acc.y);
                            acc.z = fmaf(wt, v.z, acc.z); acc.w = fmaf(wt, v.w, acc.w);
                        }
                        *reinterpret_cast<float4 *>(dst + i * pw + j) = acc;
                    }
                } else {
                    const FastDiv fd_pw(pw);
                    for (int o = tid; o < total; o += kThreads) {
                        const int i = fd_pw.div(o);
                        one(o, i, o - i * pw);
                    }
                }
            }
        }
        // with the cache, no barrier here: the H pass reads only s_t1, which the next env rewrites after its own
        // 'frame complete' barrier, and s_frame was last read before the barrier between the two passes
        if (!pcache) consumer_sync();  // s_frame is rewritten by the next env's first unit
        }
    }
}

// -------------------------------------------------------------------------- ingest: DMC
// DMCEnv._get_obs pixel/grey branch + stack logic (dmc_env.py:175-183, 193-195, 206-207,
// 228-230): 15-bit luma of the frame rendered at obs_size, pushed as is (no max-pool).
__global__ void __launch_bounds__(kThreads) k_ingest_dmc(const __grid_constant__ DevPlan p,
                                                         const uint8_t *__restrict__ f, const uint8_t *__restrict__ flags,
                                                         uint8_t *__restrict__ ring, int32_t *__restrict__ head,
                                                         float *__restrict__ pcache) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int n = blockIdx.x, tid = threadIdx.x;
    const uint8_t *src = f + (size_t)n * p.plane * 3;
    const int nvec = p.plane / 16;
    // the frame words of this thread's first two 16-pixel groups are requested before flags / head are known
    // (an idle env wastes them): one DRAM round trip per CTA instead of two
    uint32_t w0[12], w1[12];
    const int t0 = tid, t1 = tid + kThreads;
    if (t0 < nvec) {
        const uint8_t *q = src + (size_t)t0 * 48;
        *reinterpret_cast<uint4 *>(w0) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w0 + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w0 + 8) = ld_stream128(q + 32);
    }
    if (t1 < nvec) {
        const uint8_t *q = src + (size_t)t1 * 48;
        *reinterpret_cast<uint4 *>(w1) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w1 + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w1 + 8) = ld_stream128(q + 32);
    }
    const int fl = flags[n];
    const int hd = head[n];
    if (fl & AGYM_FLAG_IDLE) return;
    const int slot = (hd + 1) % p.K;
    uint8_t *s_frame = smem;
    float *s_t1 = reinterpret_cast<float *>(smem + align16(p.plane));
    __syncthreads();
    if (tid == 0) head[n] = slot;

    uint4 *dst = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + slot) * p.plane);
    const uint32_t lw01 = (2u * p.lw0) | ((2u * p.lw1) << 16), lw2 = 2u * p.lw2;
    if (t0 < nvec) {
        const uint4 o = luma16(w0, lw01, lw2);
        dst[t0] = o;
        if (pcache) reinterpret_cast<uint4 *>(s_frame)[t0] = o;
    }
    if (t1 < nvec) {
        const uint4 o = luma16(w1, lw01, lw2);
        dst[t1] = o;
        if (pcache) reinterpret_cast<uint4 *>(s_frame)[t1] = o;
    }
    for (int t = tid + 2 * kThreads; t < nvec; t += kThreads) {  // larger observations
        uint32_t w[12];
        const uint8_t *q = src + (size_t)t * 48;
        *reinterpret_cast<uint4 *>(w) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w + 8) = ld_stream128(q + 32);
        const uint4 o = luma16(w, lw01, lw2);
        dst[t] = o;
        if (pcache) reinterpret_cast<uint4 *>(s_frame)[t] = o;
    }
    if (fl & AGYM_FLAG_HARD_RESET) {
        for (int k = 0; k < p.K; ++k) {
            if (k == slot) continue;
            uint4 *z = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + k) * p.plane);
            for (int i = tid; i < p.plane / 16; i += kThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
            if (pcache) {
                float *zc = pcache + ((size_t)n * p.K + k) * p.p_h * p.p_w;
                for (int i = tid; i < p.p_h * p.p_w; i += kThreads) zc[i] = 0.f;
            }
        }
    }
    if (pcache) {
        __syncthreads();
        squeeze_to_cache(p, s_frame, s_t1, pcache + ((size_t)n * p.K + slot) * p.p_h * p.p_w, tid, kThreads);
    }
}

// ---------------------------------------------------------------------- ingest: DMC, RGB
// 16 interleaved 3-channel pixels (48 bytes, 12 words) -> the 16 bytes of each channel plane.  Output word m of
// channel c holds bytes c, 3+c, 6+c, 9+c of the 12-byte run w[3m .. 3m+2]: two PRMTs per word, no arithmetic.
__device__ __forceinline__ void split_rgb16(const uint32_t (&w)[12], uint4 &r, uint4 &g, uint4 &b) {
    uint32_t o[3][4];
#pragma unroll
    for (int m = 0; m < 4; ++m) {
        const uint32_t w0 = w[3 * m], w1 = w[3 * m + 1], w2 = w[3 * m + 2];
        o[0][m] = __byte_perm(__byte_perm(w0, w1, 0x0630), w2, 0x5210);   // bytes 0, 3, 6 | 9
        o[1][m] = __byte_perm(__byte_perm(w0, w1, 0x0741), w2, 0x6210);   // bytes 1, 4, 7 | 10
        o[2][m] = __byte_perm(__byte_perm(w0, w1, 0x0052), w2, 0x7410);   // bytes 2, 5 | 8, 11
    }
    r = make_uint4(o[0][0], o[0][1], o[0][2], o[0][3]);
    g = make_uint4(o[1][0], o[1][1], o[1][2], o[1][3]);
    b = make_uint4(o[2][0], o[2][1], o[2][2], o[2][3]);
}

// DMCEnv._get_obs pixel branch with grey=False + stack logic (dmc_env.py:122, 175-183, 228-230): the render's three
// channels, unconverted, pushed as the three planes of the next frame slot (head indexes planes, see the header).
// Same structure and flag semantics as k_ingest_dmc; the luma is replaced by a byte split.
__global__ void __launch_bounds__(kThreads) k_ingest_dmc_rgb(const __grid_constant__ DevPlan p,
                                                             const uint8_t *__restrict__ f, const uint8_t *__restrict__ flags,
                                                             uint8_t *__restrict__ ring, int32_t *__restrict__ head,
                                                             float *__restrict__ pcache) {
    constexpr int C = 3;
    extern __shared__ __align__(16) uint8_t smem[];
    const int n = blockIdx.x, tid = threadIdx.x;
    const uint8_t *src = f + (size_t)n * p.plane * 3;
    const int nvec = p.plane / 16;
    // as in k_ingest_dmc: the first two groups are requested before flags / head are known
    uint32_t w0[12], w1[12];
    const int t0 = tid, t1 = tid + kThreads;
    if (t0 < nvec) {
        const uint8_t *q = src + (size_t)t0 * 48;
        *reinterpret_cast<uint4 *>(w0) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w0 + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w0 + 8) = ld_stream128(q + 32);
    }
    if (t1 < nvec) {
        const uint8_t *q = src + (size_t)t1 * 48;
        *reinterpret_cast<uint4 *>(w1) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w1 + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w1 + 8) = ld_stream128(q + 32);
    }
    const int fl = flags[n];
    const int hd = head[n];
    if (fl & AGYM_FLAG_IDLE) return;
    const int frames = p.K / C;
    const int slot = hd / C + 1 == frames ? 0 : hd / C + 1;
    const int plane0 = C * slot;   // planes plane0 .. plane0 + 2 receive R, G, B
    const size_t vpp = (size_t)p.plane / 16;
    uint8_t *s_frame = smem;       // [C][plane] when the cache is refreshed
    float *s_t1 = reinterpret_cast<float *>(smem + C * align16(p.plane));
    __syncthreads();
    if (tid == 0) head[n] = plane0 + C - 1;

    uint4 *dst = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + plane0) * p.plane);
    uint4 *s4 = reinterpret_cast<uint4 *>(s_frame);
    const size_t svp = align16(p.plane) / 16;
    auto put = [&](int t, const uint32_t (&w)[12]) {
        uint4 r, g, b;
        split_rgb16(w, r, g, b);
        dst[t] = r; dst[vpp + t] = g; dst[2 * vpp + t] = b;
        if (pcache) { s4[t] = r; s4[svp + t] = g; s4[2 * svp + t] = b; }
    };
    if (t0 < nvec) put(t0, w0);
    if (t1 < nvec) put(t1, w1);
    for (int t = tid + 2 * kThreads; t < nvec; t += kThreads) {  // larger observations
        uint32_t w[12];
        const uint8_t *q = src + (size_t)t * 48;
        *reinterpret_cast<uint4 *>(w) = ld_stream128(q);
        *reinterpret_cast<uint4 *>(w + 4) = ld_stream128(q + 16);
        *reinterpret_cast<uint4 *>(w + 8) = ld_stream128(q + 32);
        put(t, w);
    }
    if (fl & AGYM_FLAG_HARD_RESET) {
        for (int k = 0; k < p.K; ++k) {
            if (k >= plane0 && k < plane0 + C) continue;
            uint4 *z = reinterpret_cast<uint4 *>(ring + ((size_t)n * p.K + k) * p.plane);
            for (int i = tid; i < p.plane / 16; i += kThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
            if (pcache) {
                float *zc = pcache + ((size_t)n * p.K + k) * p.p_h * p.p_w;
                for (int i = tid; i < p.p_h * p.p_w; i += kThreads) zc[i] = 0.f;
            }
        }
    }
    if (pcache) {
#pragma unroll
        for (int c = 0; c < C; ++c) {
            __syncthreads();   // c = 0: the staged planes are complete; c > 0: the previous H pass has read s_t1
            squeeze_to_cache(p, s_frame + c * align16(p.plane), s_t1,
                             pcache + ((size_t)n * p.K + plane0 + c) * p.p_h * p.p_w, tid, kThreads);
        }
    }
}

// ------------------------------------------------------------------------------- stack
// np.stack(state_buffer) (atari_env.py:143, dmc_env.py:230): oldest -> newest.
__global__ void __launch_bounds__(kThreads) k_stack(const __grid_constant__ DevPlan p, const uint8_t *__restrict__ ring,
                                                    const int32_t *__restrict__ head, uint8_t *__restrict__ out) {
    const int n = blockIdx.x;
    const int h = head[n];
    const int vpp = p.plane / 16;
    for (int k = 0; k < p.K; ++k) {
        const uint4 *src = reinterpret_cast<const uint4 *>(ring + ((size_t)n * p.K + (h + 1 + k) % p.K) * p.plane);
        uint4 *dst = reinterpret_cast<uint4 *>(out + ((size_t)n * p.K + k) * p.plane);
        for (int i = threadIdx.x; i < vpp; i += kThreads) dst[i] = __ldg(src + i);
    }
}


}  // namespace

// --------------------------------------------------------------------------- launchers
namespace {
// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda)
using EncodeTiledFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                   const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void *f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}
// frames [N][raw_h][rowb bytes] as [N][raw_h / 5][5][rowb]; box = 2 rows of R/2 consecutive periods of one env
bool encode_period5(CUtensorMap *m, const uint8_t *frames, int rowb, int raw_h, int N, int R) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    CUtensorMapDataType dt = CU_TENSOR_MAP_DATA_TYPE_UINT8;
    int esz = 1;
    if (rowb > 256) { dt = CU_TENSOR_MAP_DATA_TYPE_UINT16; esz = 2; }
    if (rowb > 512) { dt = CU_TENSOR_MAP_DATA_TYPE_UINT32; esz = 4; }
    if (rowb % (16 * 1) != 0 || rowb / esz > 256 || R % 2 != 0 || R / 2 > 256) return false;
    const cuuint64_t dims[4] = {(cuuint64_t)(rowb / esz), 5, (cuuint64_t)(raw_h / 5), (cuuint64_t)N};
    const cuuint64_t strides[3] = {(cuuint64_t)rowb, (cuuint64_t)5 * rowb, (cuuint64_t)raw_h * rowb};
    const cuuint32_t box[4] = {(cuuint32_t)(rowb / esz), 2, (cuuint32_t)(R / 2), 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    return enc(m, dt, 4, const_cast<uint8_t *>(frames), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// AGYM_NO_TM=1: contiguous bulk copies instead of the strided tensor copies in the TMA ingest kernel (A/B)
const bool g_disable_tm = getenv("AGYM_NO_TM") != nullptr;
}  // namespace

cudaError_t launch_ingest_atari(const DevPlan &p, const uint8_t *fa, const uint8_t *fb, const uint8_t *flags,
                                uint8_t *ring, int32_t *head, float *pcache, cudaStream_t st) {
    size_t smem = a16(sizeof(int32_t) * 3 * (p.S_w + p.S_h)) + a16(2 * (size_t)2 * p.S_h * p.raw_w);
    if (pcache) smem += a16(p.plane) + sizeof(float) * p.S_h * p.p_w;
    cudaError_t e;
    if (p.std_gray && !g_disable_tma && !g_disable_tm && !g_units) {   // the standard ALE geometry has its own kernel
        e = launch_ingest_gray_std(p, fa, fb, flags, ring, head, pcache, st);
        if (e != cudaErrorNotSupported) return e;
    }
    // units per env: index into the plan's span table (gray: 3 units of 28 rows; RGB: 7 units of 12 rows = two rows
    // for each of the 6 row segments of the consumer warps, and three CTAs still fit an SM)
    // With the gap-free stages of the tensor-copy path two units of 42 rows fit three CTAs per SM for gray frames
    // (7 rows for each row segment, fewer per-unit prologues): 0.239 ms instead of 0.254 ms at three units.
    const int rowb = p.raw_w * p.raw_c;
    auto pick_units = [&](int want) {
        int ui = std::min(std::max(want, 1), 8);
        while (ui > 1 && p.tma_span_rows[ui - 1] == 0) --ui;
        if (p.tma_span_rows[ui - 1] == 0)
            for (ui = 8; ui > 1 && p.tma_span_rows[ui - 1] == 0;) --ui;
        return ui;
    };
    CUtensorMap tma, tmb;
    std::memset(&tma, 0, sizeof(tma));
    std::memset(&tmb, 0, sizeof(tmb));
    auto try_tm = [&](int units) {
        const int R = p.S_h / units;
        return p.tma_period5 && !g_disable_tm && p.S_h % units == 0 && R % 2 == 0 &&
               (reinterpret_cast<uintptr_t>(fa) & 15) == 0 && (reinterpret_cast<uintptr_t>(fb) & 15) == 0 &&
               encode_period5(&tma, fa, rowb, p.raw_h, p.N, R) && encode_period5(&tmb, fb, rowb, p.raw_h, p.N, R);
    };
    int ui = pick_units(g_units ? g_units : (p.raw_c == 3 ? 7 : 2));
    bool tm = p.tma_span_rows[ui - 1] > 0 && try_tm(ui);
    if (!tm && !g_units && p.raw_c == 1) {   // contiguous copies: three units of 28 rows
        ui = pick_units(3);
        tm = p.tma_span_rows[ui - 1] > 0 && try_tm(ui);
    }
    const bool tma_ok = p.raw_c == 1 || (p.raw_c == 3 && p.fast_ingest_rgb);
    if (p.fast_ingest && tma_ok && !g_disable_tma && p.tma_span_rows[ui - 1] > 0) {
        const int units = ui, span_rows = p.tma_span_rows[ui - 1];
        const int R = p.S_h / units;
        const size_t stage = tm ? a16(2 * (2 * (((size_t)R * rowb + 127) & ~size_t(127)) + 128)) : a16(2 * ((size_t)span_rows * rowb + 16));
        const bool std_geom = p.raw_w == 160 && p.S_w == 84;
        // stages of the shared-memory ring: the gap-free gray stages of a 3-unit split are small enough for three at 3 CTAs per SM
        const int ns = (tm && std_geom && p.raw_c == 1 && units >= 3) ? 3 : 2;
        size_t fs = (tm ? 128 : 0) + ns * stage + a16(p.plane + 16) + 16 * (size_t)p.S_h + 8 * (size_t)((units + 1) & ~1);
        if (pcache) fs += sizeof(float) * ((size_t)p.S_h * p.p_w + (size_t)p.p_w * 24 + (size_t)p.p_h * p.sq_h.taps + (size_t)p.p_h);
        int dev = 0, sms = 148, occ = 1;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
#define AGYM_LAUNCH_TMA(...)                                                                                        \
    {                                                                                                               \
        if ((e = set_smem(k_ingest_atari_tma<__VA_ARGS__>, fs)) != cudaSuccess) return e;                           \
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_ingest_atari_tma<__VA_ARGS__>, kIngestThreads, fs);   \
        e = launch_pdl(k_ingest_atari_tma<__VA_ARGS__>, dim3(std::min(p.N, sms * std::max(occ, 1))), dim3(kIngestThreads), \
                       fs, st, p, fa, fb, flags, ring, head, pcache, units, span_rows, tma, tmb);                   \
        if (e != cudaSuccess) return e;                                                                             \
    }
        if (p.raw_c == 3) {
            if (std_geom && tm) AGYM_LAUNCH_TMA(480, 84, 3, true, 2)
            else if (std_geom) AGYM_LAUNCH_TMA(480, 84, 3, false, 2)
            else if (tm) AGYM_LAUNCH_TMA(0, 0, 3, true, 2)
            else AGYM_LAUNCH_TMA(0, 0, 3, false, 2)
        } else {
            if (std_geom && tm && ns == 3) AGYM_LAUNCH_TMA(160, 84, 1, true, 3)
            else if (std_geom && tm) AGYM_LAUNCH_TMA(160, 84, 1, true, 2)
            else if (std_geom) AGYM_LAUNCH_TMA(160, 84, 1, false, 2)
            else if (tm) AGYM_LAUNCH_TMA(0, 0, 1, true, 2)
            else AGYM_LAUNCH_TMA(0, 0, 1, false, 2)
        }
#undef AGYM_LAUNCH_TMA
        return cudaGetLastError();
    }
    if (p.fast_ingest) {
        size_t fs = a16((size_t)2 * p.S_h * p.raw_w + 16) + a16(p.plane + 16);
        if (pcache) fs += sizeof(float) * p.S_h * p.p_w;
        if (p.raw_c == 1) {
            if ((e = set_smem(k_ingest_atari_fast<1>, fs)) != cudaSuccess) return e;
            k_ingest_atari_fast<1><<<p.N, kThreads, fs, st>>>(p, fa, fb, flags, ring, head, pcache);
        } else {
            if ((e = set_smem(k_ingest_atari_fast<3>, fs)) != cudaSuccess) return e;
            k_ingest_atari_fast<3><<<p.N, kThreads, fs, st>>>(p, fa, fb, flags, ring, head, pcache);
        }
        return cudaGetLastError();
    }
    if (p.raw_c == 1) {
        if ((e = set_smem(k_ingest_atari<1>, smem)) != cudaSuccess) return e;
        k_ingest_atari<1><<<p.N, kThreads, smem, st>>>(p, fa, fb, flags, ring, head, pcache);
    } else {
        if ((e = set_smem(k_ingest_atari<3>, smem)) != cudaSuccess) return e;
        k_ingest_atari<3><<<p.N, kThreads, smem, st>>>(p, fa, fb, flags, ring, head, pcache);
    }
    return cudaGetLastError();
}

cudaError_t launch_ingest_dmc(const DevPlan &p, const uint8_t *f, const uint8_t *flags, uint8_t *ring, int32_t *head,
                              float *pcache, cudaStream_t st) {
    cudaError_t e;
    if (p.C == 3) {   // RGB plan: three planes per push, one CTA per env as below
        const size_t smem = pcache ? 3 * a16(p.plane) + sizeof(float) * p.S_h * p.p_w : 0;
        if ((e = set_smem(k_ingest_dmc_rgb, smem)) != cudaSuccess) return e;
        k_ingest_dmc_rgb<<<p.N, kThreads, smem, st>>>(p, f, flags, ring, head, pcache);
        return cudaGetLastError();
    }
    size_t smem = pcache ? a16(p.plane) + sizeof(float) * p.S_h * p.p_w : 0;
    if ((e = set_smem(k_ingest_dmc, smem)) != cudaSuccess) return e;
    // plain launch: programmatic dependent launch (launch_pdl) was measured slower for this grid of 8,192 short CTAs —
    // the next kernel's CTAs, let in early, sit blocked on the SM slots the later waves need (DMC step 0.071 - 0.099 ms
    // against 0.062 ms), whether the trigger is issued at the start or at the end of the CTA
    k_ingest_dmc<<<p.N, kThreads, smem, st>>>(p, f, flags, ring, head, pcache);
    return cudaGetLastError();
}

cudaError_t launch_stack(const DevPlan &p, const uint8_t *ring, const int32_t *head, uint8_t *out, cudaStream_t st) {
    k_stack<<<p.N, kThreads, 0, st>>>(p, ring, head, out);
    return cudaGetLastError();
}


}  // namespace agym
