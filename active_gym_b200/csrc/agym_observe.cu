// sm_100a kernels: fixed fovea and foveal + peripheral merge.
#include "agym_device.cuh"

namespace agym {

namespace {

// ------------------------------------------------------------------------ observe: fixed
// FixedFovealEnv._fov_step + _get_fov_state (fov_env.py:166-203).
template <int VARIANT>
__global__ void __launch_bounds__(kThreads) k_observe_fixed(const __grid_constant__ DevPlan p,
                                                            const uint8_t *__restrict__ ring,
                                                            const int32_t *__restrict__ head,
                                                            const double *__restrict__ action,
                                                            const uint8_t *__restrict__ ctrl, int32_t *__restrict__ loc,
                                                            uint8_t *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_loc[2];
    const int n = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        int r, c;
        update_loc_fixed(p, n, action, ctrl, loc, r, c);
        s_loc[0] = r; s_loc[1] = c;
    }
    __syncthreads();
    const int r0 = s_loc[0], c0 = s_loc[1];
    const int h = head[n];
    const uint8_t *env_ring = ring + (size_t)n * p.K * p.plane;

    if (VARIANT == AGYM_OUT_CROP) {
        // (K, f_h, f_w) packed; bytes gathered from the (L2-resident) ring rows
        const int per_k = p.f_h * p.f_w, total = p.K * per_k;
        const FastDiv fd_k(per_k), fd_w(p.f_w);
        uint8_t *dst = out + (size_t)n * total;
        if ((total & 3) == 0) {
            for (int t = tid; t < total / 4; t += kThreads) {
                uint32_t word = 0u;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int b = 4 * t + i;
                    const int k = fd_k.div(b), rem = b - k * per_k;
                    const int y = fd_w.div(rem), x = rem - y * p.f_w;
                    const uint8_t *src = env_ring + (size_t)((h + 1 + k) % p.K) * p.plane;
                    word |= (uint32_t)__ldg(src + (r0 + y) * p.S_w + c0 + x) << (8 * i);
                }
                reinterpret_cast<uint32_t *>(dst)[t] = word;
            }
        } else {
            for (int b = tid; b < total; b += kThreads) {
                const int k = fd_k.div(b), rem = b - k * per_k;
                const int y = fd_w.div(rem), x = rem - y * p.f_w;
                const uint8_t *src = env_ring + (size_t)((h + 1 + k) % p.K) * p.plane;
                dst[b] = __ldg(src + (r0 + y) * p.S_w + c0 + x);
            }
        }
    } else if (VARIANT == AGYM_OUT_MASK) {
        // (K, S_h, S_w): the ring word where it lies inside the fovea, zero elsewhere
        const int wpr = p.S_w / 4, wpp = p.plane / 4;
        const FastDiv fd_wpr(wpr);
        for (int k = 0; k < p.K; ++k) {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(env_ring + (size_t)((h + 1 + k) % p.K) * p.plane);
            uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)n * p.K + k) * p.plane);
            for (int t = tid; t < wpp; t += kThreads) {
                const int y = fd_wpr.div(t), x0 = 4 * (t - y * wpr);
                uint32_t m = 0u;
                if (y >= r0 && y < r0 + p.f_h) m = word_mask(x0, c0, c0 + p.f_w);
                dst[t] = m ? (__ldg(src + t) & m) : 0u;
            }
        }
    } else {
        // resize_to_full: Resize(obs_size) of the crop, W pass then H pass (fov_env.py:120,182)
        float *s_crop = reinterpret_cast<float *>(smem);
        float *s_t = s_crop + p.f_h * p.f_w;
        const int wpr = p.S_w / 4, wpp = p.plane / 4;
        const FastDiv fd_fw(p.f_w), fd_wpr(wpr);
        for (int k = 0; k < p.K; ++k) {
            const uint8_t *src = env_ring + (size_t)((h + 1 + k) % p.K) * p.plane;
            for (int i = tid; i < p.f_h * p.f_w; i += kThreads) {
                const int y = fd_fw.div(i), x = i - y * p.f_w;
                s_crop[i] = (float)__ldg(src + (r0 + y) * p.S_w + c0 + x);
            }
            __syncthreads();
            resample_w<float>(s_crop, p.f_w, s_t, p.S_w, p.f_h, p.full_w, tid, kThreads);
            __syncthreads();
            uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)n * p.K + k) * p.plane);
            for (int t = tid; t < wpp; t += kThreads) {
                const int y = fd_wpr.div(t), x0 = 4 * (t - y * wpr);
                dst[t] = resample_h_word(s_t, p.S_w, p.full_h, y, x0);
            }
            __syncthreads();
        }
    }
}

// Crop variant, one WARP per env (8 envs per CTA): a (K, f_h, f_w) observation is only a few KB, so
// a CTA per env spends its life in the latency chain loc update -> loads -> stores; here every lane
// owns ~total/128 output words whose byte gathers are all independent and in flight together.
__global__ void __launch_bounds__(kThreads) k_observe_fixed_crop_warp(const __grid_constant__ DevPlan p,
                                                                      const uint8_t *__restrict__ ring,
                                                                      const int32_t *__restrict__ head,
                                                                      const double *__restrict__ action,
                                                                      const uint8_t *__restrict__ ctrl,
                                                                      int32_t *__restrict__ loc, uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int n = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
    if (n >= p.N) return;
    int r0 = 0, c0 = 0;
    if (lane == 0) update_loc_fixed(p, n, action, ctrl, loc, r0, c0);
    r0 = __shfl_sync(0xffffffffu, r0, 0);
    c0 = __shfl_sync(0xffffffffu, c0, 0);
    const int h = head[n];
    const int per_k = p.f_h * p.f_w, words = (p.K * per_k) >> 2;
    const FastDiv fd_k(per_k), fd_w(p.f_w);
    const uint8_t *env_ring = ring + (size_t)n * p.K * p.plane + (size_t)r0 * p.S_w + c0;
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + (size_t)n * p.K * per_k);
#pragma unroll 4
    for (int t = lane; t < words; t += 32) {
        const int b = 4 * t;
        int k = fd_k.div(b), rem = b - k * per_k;
        int y = fd_w.div(rem), x = rem - y * p.f_w;
        int slot = h + 1 + k;
        slot -= slot >= p.K ? p.K : 0;
        const uint8_t *src = env_ring + (size_t)slot * p.plane + y * p.S_w;
        uint32_t word = 0u;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            word |= (uint32_t)__ldg(src + x) << (8 * i);
            if (++x == p.f_w) {  // next fovea row, possibly next frame
                x = 0;
                src += p.S_w;
                if (++y == p.f_h) {
                    y = 0;
                    ++k;
                    slot = slot + 1 == p.K ? 0 : slot + 1;
                    src = env_ring + (size_t)slot * p.plane;
                }
            }
        }
        dst[t] = word;
    }
}

// Crop variant, second version: still one warp per env, but the K windows are first staged in the warp's
// own shared-memory slice as ALIGNED words (25 independent 4-byte loads per lane instead of 85 byte loads in
// five dependent rounds: one DRAM round trip per env), and the output words are then gathered from shared
// memory through a CTA-wide table of byte offsets that is the same for every env (it only depends on K, f).
// Requires f_h * f_w % 4 == 0 is NOT needed: the table is flat over the K * f_h * f_w output bytes.
constexpr int kCropWarps = 8;
__global__ void __launch_bounds__(kCropWarps * 32) k_observe_fixed_crop_v2(const __grid_constant__ DevPlan p,
                                                                           const uint8_t *__restrict__ ring,
                                                                           const int32_t *__restrict__ head,
                                                                           const double *__restrict__ action,
                                                                           const uint8_t *__restrict__ ctrl,
                                                                           int32_t *__restrict__ loc, uint8_t *__restrict__ out,
                                                                           int nwx) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = p.K, per_k = p.f_h * p.f_w, words = (K * per_k) >> 2, rows = K * p.f_h, quads = p.S_w >> 2;
    const int stride = nwx * 4;                                   // staged bytes per window row
    uint2 *s_off = reinterpret_cast<uint2 *>(smem);               // [words] 4 x u16: staged byte offset of each output byte
    uint32_t *s_win = reinterpret_cast<uint32_t *>(smem + align16((size_t)words * 8)) + warp * rows * nwx;
    const int n = blockIdx.x * kCropWarps + warp;
    const bool valid = n < p.N;
    // the loads of the fov update go out first: their latency hides behind the table build
    LocIn li;
    li.a0 = li.a1 = 0.0; li.r = li.c = 0; li.mode = AGYM_FOV_KEEP;
    if (valid && lane == 0) li = load_loc_in(n, action, ctrl, loc);
    const int h = valid ? head[n] : 0;
    {
        const FastDiv fd_w(p.f_w);
        for (int t = tid; t < words; t += kCropWarps * 32) {
            uint32_t o[4];
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                const int idx = 4 * t + b, row = fd_w.div(idx), x = idx - row * p.f_w;  // row = k * f_h + y
                o[b] = (uint32_t)(row * stride + x);
            }
            s_off[t] = make_uint2(o[0] | (o[1] << 16), o[2] | (o[3] << 16));
        }
    }
    int r0 = 0, c0 = 0;
    if (valid && lane == 0) {
        apply_loc(p, li, r0, c0);
        loc[2 * n] = r0;
        loc[2 * n + 1] = c0;
    }
    r0 = __shfl_sync(0xffffffffu, r0, 0);
    c0 = __shfl_sync(0xffffffffu, c0, 0);
    const int wq0 = c0 >> 2, cb = c0 & 3;
    if (valid) {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(ring) + (size_t)n * K * (p.plane >> 2) + r0 * quads + wq0;
        const FastDiv fd_n(nwx), fd_h(p.f_h);
        const int wmax = quads - 1 - wq0;   // last word of a frame row: the spare staged word must not run past the ring
#pragma unroll 4
        for (int i = lane; i < rows * nwx; i += 32) {
            const int row = fd_n.div(i), w = i - row * nwx;
            const int k = fd_h.div(row), y = row - k * p.f_h;
            int slot = h + 1 + k;
            slot -= slot >= K ? K : 0;
            cp_async4(s_win + i, src + slot * (p.plane >> 2) + y * quads + min(w, wmax));
        }
    }
    cp_async_commit();
    __syncthreads();   // offset table complete
    if (!valid) return;
    cp_async_wait<0>();
    __syncwarp();
    const uint8_t *wb = reinterpret_cast<const uint8_t *>(s_win) + cb;
    uint32_t *dst = reinterpret_cast<uint32_t *>(out + (size_t)n * K * per_k);
#pragma unroll 4
    for (int t = lane; t < words; t += 32) {
        const uint2 o = s_off[t];
        const uint32_t b0 = wb[o.x & 0xffffu], b1 = wb[o.x >> 16], b2 = wb[o.y & 0xffffu], b3 = wb[o.y >> 16];
        const uint32_t word = __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
        dst[t] = word;
        if (p.norm_out) norm_store4(p.norm_dt, word, p.norm_out, (size_t)n * words + t);   // uniform branch
    }
}

// Crop variant, third version.  One warp per env as before, but (i) the window rows are staged as their 16-byte-aligned
// hulls by 16-byte cp.async (a lane takes whole rows: 3 copies per 30-pixel row instead of 9 four-byte copies, each with
// its own index arithmetic), (ii) a lane assembles the output words of a GROUP of g rows (g * f_w bytes = whole words:
// g = 1, 2 or 4) by funnel-shifting the aligned words of each row — one LDS + one SHF per output word instead of a table
// load, four byte loads and three PRMTs — and parks them in a shared-memory tile that holds the CTA's envs back to back,
// (iii) the tile leaves as ONE TMA bulk store per CTA (4 or 8 envs are a multiple of 16 bytes whatever the window), or as
// coalesced words from the last, partial CTA.  F_W != 0 fixes the window width at compile time (every loop unrolls, no
// per-word bookkeeping); F_W == 0 is the same code for any width.  Measured (DESIGN.md 3.5): the crop is bound by its
// scattered 64-byte DRAM granules, not by instructions — v3 is 4-9 % faster than v2 away from 8,192 envs, equal there.
struct CropV3Args {
    int nch;                // 16-byte chunks per staged row: (f_w + 30) / 16
    int g, gw, ngroups;     // rows / output words per group, groups per env
    uint32_t m_fh;          // FastDiv multiplier of f_h (host-computed)
    int slice;              // staged bytes per warp (incl. 16 spare bytes in front)
};
constexpr int kCrop3Warps = 8;
template <int F_W, int WARPS = kCrop3Warps>   // WARPS: envs per CTA
__global__ void __launch_bounds__(WARPS * 32) k_observe_fixed_crop_v3(const __grid_constant__ DevPlan p,
                                                                            const uint8_t *__restrict__ ring,
                                                                            const int32_t *__restrict__ head,
                                                                            const double *__restrict__ action,
                                                                            const uint8_t *__restrict__ ctrl,
                                                                            int32_t *__restrict__ loc, uint8_t *__restrict__ out,
                                                                            const CropV3Args a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = blockIdx.x * WARPS + warp;
    const bool valid = n < p.N;
    const int fw = F_W ? F_W : p.f_w;
    const int nch = F_W ? (F_W + 30) / 16 : a.nch;
    const int g = F_W ? (F_W % 4 == 0 ? 1 : F_W % 2 == 0 ? 2 : 4) : a.g;
    const int gw = g * fw / 4;
    const int K = p.K, rows = K * p.f_h, stride = nch * 16, out_env = rows * fw, words = out_env >> 2;
    uint8_t *s_in = smem + (size_t)warp * a.slice + 16;   // [rows][stride]; 16 spare bytes in front (a row's first word may start 3 bytes early)
    uint32_t *s_tile = reinterpret_cast<uint32_t *>(smem + (size_t)WARPS * a.slice);   // [envs of the CTA][words]
    uint32_t *s_out = s_tile + warp * words;
    if (valid) {
        LocIn li;
        li.a0 = li.a1 = 0.0; li.r = li.c = 0; li.mode = AGYM_FOV_KEEP;
        if (lane == 0) li = load_loc_in(n, action, ctrl, loc);
        const int h = head[n];
        int r0 = 0, c0 = 0;
        if (lane == 0) {
            apply_loc(p, li, r0, c0);
            loc[2 * n] = r0;
            loc[2 * n + 1] = c0;
        }
        r0 = __shfl_sync(0xffffffffu, r0, 0);
        c0 = __shfl_sync(0xffffffffu, c0, 0);
        const FastDiv fd_h(p.f_h, a.m_fh);
        const int first0 = r0 * p.S_w + c0;   // byte offset of the window's first pixel in a plane
        const uint8_t *env = ring + (size_t)n * K * p.plane;
        for (int row = lane; row < rows; row += 32) {
            const int k = fd_h.div(row), y = row - k * p.f_h;
            int slot = h + 1 + k;
            slot -= slot >= K ? K : 0;
            const int first = first0 + y * p.S_w, lead = first & 15;
            const uint8_t *src = env + (size_t)slot * p.plane + (first - lead);
            const uint32_t dst = smem_u32(s_in + row * stride);
            // a chunk past the row's last pixel is not needed (and may lie behind the ring's end)
            if (F_W) {
#pragma unroll
                for (int j = 0; j < (F_W + 30) / 16; ++j)
                    if (16 * j < lead + fw) cp_async16_s(dst + 16 * j, src + 16 * j);
            } else {
                for (int j = 0; j < nch; ++j)
                    if (16 * j < lead + fw) cp_async16_s(dst + 16 * j, src + 16 * j);
            }
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
        for (int grp = lane; grp < a.ngroups; grp += 32) {
            uint32_t carry = 0u;
            uint32_t *dstw = s_out + grp * gw;
            if (F_W) {
                constexpr int G = F_W % 4 == 0 ? 1 : F_W % 2 == 0 ? 2 : 4;
#pragma unroll
                for (int i = 0; i < G; ++i) {
                    constexpr int FW = F_W ? F_W : 4;
                    const int ob = i * FW, s = ob & 3, w0 = ob >> 2, w1 = (ob + FW - 1) >> 2;
                    const bool open_end = ((ob + FW) & 3) != 0;
                    const int row = grp * G + i, k = fd_h.div(row), y = row - k * p.f_h;
                    const int src = row * stride + ((first0 + y * p.S_w) & 15) - s;
                    const uint32_t sh = (uint32_t)(src & 3) * 8u;
                    const uint32_t *wp = reinterpret_cast<const uint32_t *>(s_in + (src & ~3));
                    uint32_t prev = wp[0];
#pragma unroll
                    for (int w = w0; w <= w1; ++w) {
                        const uint32_t next = wp[w - w0 + 1];
                        uint32_t v = __funnelshift_r(prev, next, sh);
                        prev = next;
                        if (w == w0 && s) {
                            const uint32_t m = (1u << (8 * s)) - 1u;
                            v = (carry & m) | (v & ~m);
                        }
                        if (w == w1 && open_end) carry = v;
                        else dstw[w] = v;
                    }
                }
            } else {
                int ob = 0;   // byte offset of the current row inside the group's output
                for (int i = 0; i < g; ++i, ob += fw) {
                    const int row = grp * g + i, k = fd_h.div(row), y = row - k * p.f_h;
                    const int s = ob & 3;                                             // bytes of the first word that belong to the row before
                    const int src = row * stride + ((first0 + y * p.S_w) & 15) - s;   // staged byte that lands in byte 0 of that word (>= -3)
                    const uint32_t sh = (uint32_t)(src & 3) * 8u;
                    const uint32_t *wp = reinterpret_cast<const uint32_t *>(s_in + (src & ~3));
                    const int w0 = ob >> 2, w1 = (ob + fw - 1) >> 2;
                    const bool open_end = ((ob + fw) & 3) != 0;                       // the last word is finished by the next row
                    uint32_t prev = wp[0];
                    for (int w = w0; w <= w1; ++w) {
                        const uint32_t next = wp[w - w0 + 1];
                        uint32_t v = __funnelshift_r(prev, next, sh);
                        prev = next;
                        if (w == w0 && s) {
                            const uint32_t m = (1u << (8 * s)) - 1u;
                            v = (carry & m) | (v & ~m);
                        }
                        if (w == w1 && open_end) carry = v;
                        else dstw[w] = v;
                    }
                }
            }
        }
    }
    const int n0 = blockIdx.x * WARPS;
    const bool bulk = n0 + WARPS <= p.N && (reinterpret_cast<uintptr_t>(out) & 15) == 0;   // uniform over the CTA
    if (bulk) {
        fence_async_smem();
        __syncthreads();
        if (threadIdx.x == 0) {
            bulk_s2g(out + (size_t)n0 * out_env, s_tile, (uint32_t)(WARPS * out_env));
            bulk_commit();
        }
    } else if (valid) {
        __syncwarp();
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + (size_t)n * out_env);
        for (int t = lane; t < words; t += 32) dst[t] = s_out[t];
    }
    if (p.norm_out && valid) {   // the normalised copy of the same tile
        __syncwarp();
        for (int t = lane; t < words; t += 32) norm_store4(p.norm_dt, s_out[t], p.norm_out, (size_t)n * words + t);
    }
    if (bulk && threadIdx.x == 0) bulk_wait_read<0>();   // shared memory must outlive the store's reads
}

// ------------------------------------------------------------------- observe: peripheral
// FixedFovealPeripheralEnv._get_fov_state (fov_env.py:375-388):
//   out = Resize(obs)(Resize(peripheral_res)(full)); out[fovea] = full[fovea].
// CACHED: the squeeze of every ring slot was stored at ingest time (it does not depend on
// fov_loc), so only the expand + paste remain per step.
template <bool CACHED>
__global__ void __launch_bounds__(kThreads) k_observe_peripheral(const __grid_constant__ DevPlan p,
                                                                 const uint8_t *__restrict__ ring,
                                                                 const int32_t *__restrict__ head,
                                                                 const float *__restrict__ pcache,
                                                                 const double *__restrict__ action,
                                                                 const uint8_t *__restrict__ ctrl,
                                                                 int32_t *__restrict__ loc, uint8_t *__restrict__ out) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_loc[2];
    const int n = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) {
        int r, c;
        update_loc_fixed(p, n, action, ctrl, loc, r, c);
        s_loc[0] = r; s_loc[1] = c;
    }
    __syncthreads();
    const int r0 = s_loc[0], c0 = s_loc[1];
    const int h = head[n];

    // shared: frame u8 [plane] | t1 f32 [S_h][p_w] | sq f32 [p_h][p_w] | t2 f32 [p_h][S_w]
    uint8_t *s_frame = smem;
    float *s_t1 = reinterpret_cast<float *>(smem + align16(p.plane));
    float *s_sq = s_t1 + p.S_h * p.p_w;
    float *s_t2 = s_sq + p.p_h * p.p_w;
    const int wpr = p.S_w / 4, wpp = p.plane / 4;
    const FastDiv fd_wpr(wpr);

    for (int k = 0; k < p.K; ++k) {
        const int slot = (h + 1 + k) % p.K;
        const uint8_t *src = ring + ((size_t)n * p.K + slot) * p.plane;
        if (!CACHED) {
            for (int i = tid; i < p.plane / 16; i += kThreads)
                reinterpret_cast<uint4 *>(s_frame)[i] = __ldg(reinterpret_cast<const uint4 *>(src) + i);
            __syncthreads();
            resample_w<uint8_t>(s_frame, p.S_w, s_t1, p.p_w, p.S_h, p.sq_w, tid, kThreads);
            __syncthreads();
            resample_h<float>(s_t1, p.p_w, s_sq, p.p_w, p.p_w, p.sq_h, tid, kThreads);
            __syncthreads();
        } else {
            const float *c = pcache + ((size_t)n * p.K + slot) * p.p_h * p.p_w;
            for (int i = tid; i < p.p_h * p.p_w; i += kThreads) s_sq[i] = __ldg(c + i);
            __syncthreads();
        }
        resample_w<float>(s_sq, p.p_w, s_t2, p.S_w, p.p_h, p.ex_w, tid, kThreads);
        __syncthreads();
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + ((size_t)n * p.K + k) * p.plane);
        const uint32_t *sharp_g = reinterpret_cast<const uint32_t *>(src);
        const uint32_t *sharp_s = reinterpret_cast<const uint32_t *>(s_frame);
        for (int t = tid; t < wpp; t += kThreads) {
            const int y = fd_wpr.div(t), x0 = 4 * (t - y * wpr);
            uint32_t v = resample_h_word(s_t2, p.S_w, p.ex_h, y, x0);
            if (y >= r0 && y < r0 + p.f_h) {
                const uint32_t m = word_mask(x0, c0, c0 + p.f_w);
                if (m) v = (v & ~m) | ((CACHED ? __ldg(sharp_g + t) : sharp_s[t]) & m);
            }
            dst[t] = v;
        }
        __syncthreads();
    }
}

// Fast peripheral observe (cached squeeze, bilinear-upsample expand): both expand passes are
// two-tap lerps r = b + w0 * (a - b).  The cached squeeze is biased by kBias on load (see agym_device.cuh).


// Persistent CTAs (a few per SM) walk the env batch.  Per env:
//   prefetch  the cached squeeze of its K ring slots and the ring words under its fovea arrive by
//             cp.async into a double buffer, one env ahead of the arithmetic; thread 0 also applies
//             the NEXT-but-one env's sensory action to fov_loc (fov_env.py:187-199), so no separate
//             launch is needed and the prefetch knows where the fovea will be;
//   phase A   W-expand: T[k][j][x] = w0[x]*sq[k][j][i0[x]] + w1[x]*sq[k][j][i0[x]+1] + bias for the
//             K*p_h squeezed rows, two columns per thread (FFMA2), kept in shared memory;
//   phase B   H-expand + quantise + paste: one thread owns 4 adjacent columns and a segment of
//             output rows for KG frames; it holds rows b = T[j0+1] and d = T[j0]-T[j0+1] in
//             registers (reloaded only when the source row changes, ~every 4th output row) and
//             emits one 4-pixel word per frame and row: 2 FFMA2 + 3 PRMT + 1 STG.
// The bias 49152.5 makes the rounded pixel floor(v + 0.5) appear in byte 1 of the float's bit
// pattern (ulp there is 2^-8: total evaluation error < 0.01 u8 LSB), so quantisation needs no
// float->int conversion.
template <int KG, int PW>  // KG: frames per thread (K % KG == 0); PW: words per plane if known at compile time, else 0
__global__ void __launch_bounds__(128) k_observe_peripheral_v2(const __grid_constant__ DevPlan p,
                                                               const uint8_t *__restrict__ ring,
                                                               const int32_t *__restrict__ head,
                                                               const float *__restrict__ pcache,
                                                               const double *__restrict__ action,
                                                               const uint8_t *__restrict__ ctrl,
                                                               int32_t *__restrict__ loc, uint8_t *__restrict__ out,
                                                               int ysegs) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int s_loc[2][2];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int pp = p.p_h * p.p_w, K = p.K, N = p.N, f_h = p.f_h, S_w = p.S_w;
    const int quads = S_w >> 2;
    const uint32_t wpp = PW ? (uint32_t)PW : ((uint32_t)p.plane >> 2);  // words per plane
    const int nw_max = (p.f_w + 3) / 4 + 1;
    const int sq_words = (K * pp + 3) & ~3, buf_words = sq_words + ((K * f_h * nw_max + 3) & ~3);
    const int trows = K * p.p_h;
    float *bufs = reinterpret_cast<float *>(smem);  // [2]{ sq [K][p_h][p_w] | fov [K][f_h][nw_max] }
    float *s_T = bufs + 2 * buf_words;              // [K * p_h][S_w], biased
    int2 *s_row = reinterpret_cast<int2 *>(s_T + trows * S_w);  // [S_h + 1] {source row j0, bits of w0}
    const uint32_t *ring_w = reinterpret_cast<const uint32_t *>(ring);
    uint32_t *out_w = reinterpret_cast<uint32_t *>(out);
    const int G = gridDim.x;

    // ---- per-thread constants
    // phase A: column pair cp, rows part, part + parts, ...
    const int npairs = S_w >> 1, parts = nt / npairs;
    const int a_part = tid / npairs, cp = tid - a_part * npairs;
    const bool a_active = a_part < parts;
    int a_i0 = 0, a_i1 = 0;
    uint64_t a_w0 = 0, a_w1 = 0;
    if (a_active) {
        a_i0 = __ldg(p.exw_i0 + 2 * cp);
        a_i1 = __ldg(p.exw_i0 + 2 * cp + 1);
        a_w0 = pack2(__ldg(p.exw_w0 + 2 * cp), __ldg(p.exw_w0 + 2 * cp + 1));
        a_w1 = pack2(__ldg(p.exw_w1 + 2 * cp), __ldg(p.exw_w1 + 2 * cp + 1));
    }
    const uint64_t bias2 = pack2(kBias, kBias);
    // phase B: column quad q, row segment g
    const int g = tid / quads, q = tid - g * quads;
    const bool active = g < ysegs;
    const int rows_per = (p.S_h + ysegs - 1) / ysegs;
    const int y_begin = g * rows_per, y_end = active ? min(p.S_h, y_begin + rows_per) : y_begin;
    const int pp4 = pp >> 2, frows = K * f_h;
    for (int i = tid; i < p.S_h; i += nt) s_row[i] = make_int2(__ldg(p.exh_i0 + i), __float_as_int(__ldg(p.exh_w0 + i)));
    if (tid == 0) s_row[p.S_h] = make_int2(-1, 0);  // sentinel: ends the last run of rows

    auto issue = [&](int env, int lr, int lc, int hh, int b) {
        float *sq = bufs + b * buf_words;
        uint32_t *fv = reinterpret_cast<uint32_t *>(sq + sq_words);
        const size_t slot0 = (size_t)env * K;
        for (int k = 0; k < K; ++k) {  // cached squeeze: logical frame k <- ring slot (hh+1+k)%K
            int slot = hh + 1 + k;
            slot -= slot >= K ? K : 0;
            const float *src = pcache + (slot0 + slot) * pp;
            for (int c = tid; c < pp4; c += nt) cp_async16(sq + k * pp + 4 * c, src + 4 * c);
        }
        const int wq0 = lc >> 2, nw = ((lc + p.f_w - 1) >> 2) - wq0 + 1;
        for (int r = tid; r < frows; r += nt) {  // one fovea row (k, yy) per thread and pass
            const int k = r / f_h, yy = r - k * f_h;
            int slot = hh + 1 + k;
            slot -= slot >= K ? K : 0;
            const uint32_t *src = ring_w + (slot0 + slot) * wpp + (uint32_t)(lr + yy) * quads + wq0;
            uint32_t *dst = fv + r * nw_max;
            for (int w = 0; w < nw; ++w) cp_async4(dst + w, src + w);
        }
    };
    // fov_loc of env `env` after this step's sensory action; thread 0 only
    auto next_loc = [&](int env, int slot) {
        int r = 0, c = 0;
        if (env < N) update_loc_fixed<true>(p, env, action, ctrl, loc, r, c);
        s_loc[slot][0] = r;
        s_loc[slot][1] = c;
    };

    int e = blockIdx.x;
    if (tid == 0) { next_loc(e, 0); next_loc(e + G, 1); }
    __syncthreads();
    int lr = s_loc[0][0], lc = s_loc[0][1], lr1 = s_loc[1][0], lc1 = s_loc[1][1];
    int hh = 0, hh1 = 0;
    if (e < N) { hh = head[e]; issue(e, lr, lc, hh, 0); }
    cp_async_commit();
    if (e + G < N) hh1 = head[e + G];
    __syncthreads();  // s_loc is rewritten below

    for (int it = 0; e < N; e += G, ++it) {
        const int en = e + G;
        if (en < N) issue(en, lr1, lc1, hh1, (it + 1) & 1);
        cp_async_commit();
        if (tid == 0) next_loc(en + G, it & 1);
        int hh2 = 0;
        if (en + G < N) hh2 = head[en + G];
        cp_async_wait<1>();
        __syncthreads();

        const float *sq = bufs + (it & 1) * buf_words;
        // ---- phase A: W-expand every squeezed row into s_T
        if (a_active) {
            const float *s = sq + a_part * p.p_w;
            float *t = s_T + a_part * S_w + 2 * cp;
            const int sstep = parts * p.p_w, tstep = parts * S_w;
#pragma unroll 4
            for (int r = a_part; r < trows; r += parts, s += sstep, t += tstep) {
                const uint64_t u = pack2(s[a_i0], s[a_i1]), v = pack2(s[a_i0 + 1], s[a_i1 + 1]);
                *reinterpret_cast<uint64_t *>(t) = ffma2(a_w0, u, ffma2(a_w1, v, bias2));
            }
        }
        __syncthreads();

        // ---- phase B: H-expand, quantise, paste the fovea, store
        if (active) {
            const uint32_t *fvb = reinterpret_cast<const uint32_t *>(sq + sq_words);
            const uint32_t fov_mask = word_mask(4 * q, lc, lc + p.f_w);
            const int rf = fov_mask ? lr : (1 << 29);  // this column quad never meets the fovea
            const int fstride = f_h * nw_max;          // words between two frames' fovea tiles
            for (int k0 = 0; k0 < K; k0 += KG) {
                uint32_t *orow = out_w + ((size_t)e * K + k0) * wpp + (uint32_t)y_begin * quads + q;
                const uint32_t *fv = fvb + (k0 * f_h - rf) * nw_max + (q - (lc >> 2));
                const float *tk = s_T + (size_t)k0 * p.p_h * S_w + 4 * q;
                const int kstride = p.p_h * S_w;
                int y = y_begin, j_have = -2;
                const int2 *rp = s_row + y_begin;
                int2 rw = *rp;
                uint64_t b0[KG], b1[KG], d0[KG], d1[KG];
                while (y < y_end) {
                    const int j0 = rw.x;
#pragma unroll
                    for (int kk = 0; kk < KG; ++kk) {
                        const float *tj = tk + kk * kstride + j0 * S_w;
                        uint64_t a0, a1;
                        if (j0 == j_have + 1) { a0 = b0[kk]; a1 = b1[kk]; }
                        else { const ulonglong2 a = *reinterpret_cast<const ulonglong2 *>(tj); a0 = a.x; a1 = a.y; }
                        const ulonglong2 b = *reinterpret_cast<const ulonglong2 *>(tj + S_w);
                        b0[kk] = b.x; b1[kk] = b.y;
                        d0[kk] = fsub2(a0, b.x); d1[kk] = fsub2(a1, b.y);
                    }
                    j_have = j0;
                    do {
                        const float w0 = __int_as_float(rw.y);
                        const uint64_t w2 = pack2(w0, w0);
                        rw = *++rp;  // next output row (sentinel past the end)
                        uint32_t word[KG];
#pragma unroll
                        for (int kk = 0; kk < KG; ++kk) {
                            uint32_t u0, u1, u2, u3;
                            unpack2(ffma2(w2, d0[kk], b0[kk]), u0, u1);
                            unpack2(ffma2(w2, d1[kk], b1[kk]), u2, u3);
                            word[kk] = __byte_perm(__byte_perm(u0, u1, 0x0051), __byte_perm(u2, u3, 0x0051), 0x5410);
                        }
                        if ((unsigned)(y - rf) < (unsigned)f_h) {  // fovea rows: paste the sharp bytes (fov_env.py:385-386)
                            const uint32_t *sh = fv + y * nw_max;
#pragma unroll
                            for (int kk = 0; kk < KG; ++kk) word[kk] = (word[kk] & ~fov_mask) | (sh[kk * fstride] & fov_mask);
                        }
#pragma unroll
                        for (int kk = 0; kk < KG; ++kk) orow[kk * wpp] = word[kk];
                        orow += quads;
                        ++y;
                    } while (rw.x == j0 && y < y_end);
                }
            }
        }
        __syncthreads();  // s_T, s_loc and the buffer just read are rewritten next
        lr = lr1; lc = lc1; hh = hh1; hh1 = hh2;
        lr1 = s_loc[it & 1][0]; lc1 = s_loc[it & 1][1];
    }
}

// Standard geometry (obs 84x84, periphery 20x20): the H-expand pattern is known at compile time —
// output row y = 21 g + r reads squeezed rows 5 g - 1 + t(r), 5 g + t(r) with t(r) = src(r) + 1
// (clamped at the frame border) — so the row loop is fully unrolled: register-resident rows,
// immediate offsets, no index arithmetic.  The plan checks the host tables against this pattern
// before the kernel is used; the WEIGHTS always come from the host tables (ATen's values).
//
// One thread = one 4-pixel column quad q of one frame k over one 21-row segment g (21 x 4 threads
// per plane).  It W-expands the 7 squeezed rows it needs straight from the cached squeeze
// in shared memory — three adjacent samples s0..s2 cover its four columns, so
//   T[c] = a[c] * s0 + b[c] * s1 + g[c] * s2 + bias      (one of a[c], g[c] is zero)
// is 6 FFMA2 per row with per-thread constant weights — then H-expands, quantises, pastes the
// fovea and stores one word per row: 2 FFMA2 + 3 PRMT + (LDS + LOP3 on fovea rows) + 1 STS.
// The bias 49152.5 puts the rounded pixel floor(v + 0.5) into byte 1 of the float (ulp 2^-8,
// total evaluation error < 0.01 u8 LSB), so there is no float->int conversion.
//
// Persistent CTAs of K plane groups: group k (3 warps, 96 threads, 84 of them computing) produces
// frame k of every env of the CTA and runs its own pipeline, synchronised by its own named barrier —
// there is no CTA-wide barrier in the env loop, so a thread waits only for the 95 others that share
// its plane and a group may run ahead of the others by the depth of its own buffers.  Per group:
//   - inputs run two envs ahead through three shared-memory buffers: for env e+2 the group's
//     leader issues one TMA bulk copy (cp.async.bulk, completion on the group's own mbarrier) of the
//     plane's cached squeeze (400 f32), and the group stages its plane's fovea bytes itself (below),
//     so the copies it waits for are its own;
//   - the plane is assembled in a double-buffered 7,056-byte tile and leaves as ONE TMA bulk store
//     to out + e * 28,224 + k * 7,056 (4-byte stores straight to global ran the write path at 40 %
//     of HBM bandwidth); the leader issues, commits and waits its group's bulk groups, which are
//     per thread, so the groups do not interfere.
// The sensory actions: every 32 iterations warp 0 applies those of the CTA's next 32 envs to fov_loc,
// one env per lane (fov_env.py:187-199), into a ring of four 32-entry batches.  A batch is published
// on its `loc_full` mbarrier (the groups wait for it before they prefetch its first env) and handed
// back on its `loc_free` mbarrier (each group's leader arrives once the group has left the batch), so
// warp 0 rewrites a slot only after every group has passed it, however far apart the groups run.
struct StdGeom {
    static constexpr int S = 84, P = 20, Q = 21, SEG = 4, R = 21, SPAN = 7;
    // floor((40 i - 64) / 168): source index of output i relative to the 20-sample axis
    __host__ __device__ static constexpr int src(int i) { return (40 * i - 64 + 168 * 4) / 168 - 4; }
};

// rows r of a 21-row segment whose bit is set in `rows`: stage ring word (row r, this quad) at fovea-tile row r
template <int NW, int R0>
__device__ __forceinline__ void prefetch_rows_imm(uint32_t rows, uint32_t dst, const uint32_t *src) {
    if constexpr (R0 < StdGeom::R) {
        if (rows & (1u << R0)) cp_async4_imm<R0 * (NW ? NW : 1) * 4, R0 * StdGeom::Q * 4>(dst, src);
        prefetch_rows_imm<NW, R0 + 1>(rows, dst, src);
    }
}

// FS ("full-row staging"): the sharp fovea bytes are staged as 16-byte chunks at the positions they have in the ring
// (the staging buffer of a frame mirrors the ring words [lr * 21 & ~3, ...) of its slot, so a chunk copy is aligned on
// both sides and the paste reads word (row r, quad q) at an immediate offset).  Only the chunks that meet the fovea
// columns are copied: f_h * 3 copies of 16 bytes per plane, about one per thread of the plane's group and a dozen
// instructions each, instead of up to 21 predicated 4-byte copies per thread (a quarter of the kernel's instructions).
// A chunk is pasted by other threads than the one that copied it, so each group copies its own plane's chunks and
// waits for them before its own barrier.  Costs 2.5 KB of shared memory per frame and buffer; used when two CTAs
// still fit an SM (the standard 30x30 fovea does).
template <int K, int NW, bool FS>  // NW: words per staged fovea row, (f_w + 3) / 4 + 1, when baked in; 0 = from the plan
__global__ void __launch_bounds__(96 * K, 2)
    k_observe_peripheral_std(const __grid_constant__ DevPlan p, const __grid_constant__ ExpandStd ew,
                             const uint8_t *__restrict__ ring, const int32_t *__restrict__ head,
                             const float *__restrict__ pcache, const double *__restrict__ action,
                             const uint8_t *__restrict__ ctrl, int32_t *__restrict__ loc, uint8_t *__restrict__ out) {
    using Gm = StdGeom;
    constexpr int S = Gm::S, P = Gm::P, Q = Gm::Q, R = Gm::R;
    constexpr int GT = 96;  // threads of one plane group
    constexpr int PP = P * P, PLANE_W = S * S / 4;
    constexpr int NBUF = 3, DIST = 2, LOC_RING = 128, LOC_BATCHES = LOC_RING / 32;
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ int4 s_loc[LOC_RING];  // {fov row, fov col, head, -} of the CTA's iteration j at [j % LOC_RING]
    __shared__ __align__(8) uint64_t full[K][NBUF];
    __shared__ __align__(8) uint64_t loc_full[LOC_BATCHES], loc_free[LOC_BATCHES];
    const int tid = threadIdx.x;
    const int k = tid / GT, lt = tid - k * GT;  // plane group = frame k of the stack; thread lt of the group
    const bool lead = lt == 0;
    const int N = p.N, f_h = p.f_h, f_w = p.f_w, G = gridDim.x;
    const int nw_max = NW ? NW : (f_w + 3) / 4 + 1;
    const int rowbuf = (f_h * Q + 9) & ~3;  // FS: staged words of one frame (alignment slack on both sides)
    const int buf_words = PP + (FS ? rowbuf : ((f_h * nw_max + 3) & ~3));
    // the group's shared memory: [NBUF]{ sq [P][P] | fov [f_h][nw_max] or [rowbuf] }, then [2][S][S / 4] output words
    float *bufs = reinterpret_cast<float *>(smem) + k * (NBUF * buf_words + 2 * PLANE_W);
    uint32_t *tiles = reinterpret_cast<uint32_t *>(bufs + NBUF * buf_words);
    const uint32_t *ring_w = reinterpret_cast<const uint32_t *>(ring);

    // fov_loc (after this step's action) and head of iterations [it0, it0 + 32), one per lane (warp 0)
    auto loc_batch = [&](int it0) {
        const int bt = it0 / 32;
        if (bt >= LOC_BATCHES) mbar_wait(&loc_free[bt % LOC_BATCHES], (bt / LOC_BATCHES - 1) & 1);  // every group left bt - 4
        const int j = it0 + (tid & 31);
        // j * G cannot overflow: a CTA runs at most N / G + 1 iterations and batches reach 64 past that
        const int env = j <= N / G + 1 ? (int)blockIdx.x + j * G : N;
        int r = 0, c = 0, hh = 0;
        if (env < N) {
            update_loc_fixed<true>(p, env, action, ctrl, loc, r, c);
            hh = head[env];
        }
        s_loc[j & (LOC_RING - 1)] = make_int4(r, c, hh, 0);
        mbar_arrive(&loc_full[bt % LOC_BATCHES]);
    };
    pdl_launch_dependents();
    if (tid == 0) {
        for (int i = 0; i < K * NBUF; ++i) mbar_init(&full[i / NBUF][i % NBUF], 1);
        for (int i = 0; i < LOC_BATCHES; ++i) {
            mbar_init(&loc_full[i], 32);
            mbar_init(&loc_free[i], K);
        }
        mbar_fence_init();
    }

    const bool active = lt < Q * Gm::SEG;
    // segment order 3, 0, 1, 2 over the group's runs of 21 threads: of the tile stores (word 441 g + 21 r + q), only
    // the middle warp's are 2-way bank conflicts; in order 0..3 two of the three warps had them
    const int q = lt % Q, g = (lt / Q + 3) & 3;
    // W pass: samples base .. base + 2 of a squeezed row cover this quad's columns
    int base;
    uint64_t wa01, wa23, wb01, wb23, wc01, wc23;  // weights of s0 / s1 / s2 for columns (0,1) and (2,3)
    {
        const int i00 = __ldg(p.exw_i0 + 4 * q);
        base = min(i00, P - 3);
        float wa[4], wb[4], wc[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int sel = __ldg(p.exw_i0 + 4 * q + c) - base;  // 0 or 1
            const float w0 = __ldg(p.exw_w0 + 4 * q + c), w1 = __ldg(p.exw_w1 + 4 * q + c);
            wa[c] = sel == 0 ? w0 : 0.f;
            wb[c] = sel == 0 ? w1 : w0;
            wc[c] = sel == 0 ? 0.f : w1;
        }
        wa01 = pack2(wa[0], wa[1]); wa23 = pack2(wa[2], wa[3]);
        wb01 = pack2(wb[0], wb[1]); wb23 = pack2(wb[2], wb[3]);
        wc01 = pack2(wc[0], wc[1]); wc23 = pack2(wc[2], wc[3]);
    }
    const uint64_t bias2 = pack2(kBias, kBias);
    // squeezed rows 5g-1 .. 5g+5, clamped to the frame: float offsets inside one staged squeeze
    const int row_first = 5 * g - 1;
    const int so_t0 = (row_first < 0 ? 0 : row_first) * P + base;                 // t = 0
    const int so_mid = row_first * P + base;                                      // t = 1..5 at + t * P
    const int so_t6 = (row_first + 6 > P - 1 ? P - 1 : row_first + 6) * P + base;  // t = 6
    const uint32_t bufs_s = smem_u32(bufs);
    const uint32_t word0 = (uint32_t)(g * R) * Q + q;  // this thread's first output word inside a plane
    // FS: the (at most two) 16-byte chunks this thread stages of its plane for every env: chunk c of fovea row y
    // (the launcher's bound on K * f_h * chunks per row keeps a plane within 2 * 96 chunks)
    constexpr int NJ = 2;
    int ck_row[NJ], ck_c4[NJ];
    if constexpr (FS) {
        const int cpr = (f_w + 14) / 16 + 1, total = f_h * cpr;
#pragma unroll
        for (int a = 0; a < NJ; ++a) {
            const int i = lt + a * GT, row = i / cpr;
            ck_row[a] = i < total ? row * Q : -1;
            ck_c4[a] = (i - row * cpr) * 4;
        }
    }

    // one bit per row r of this segment that meets the fovea at (lr, lc); 0 if the quad misses it
    auto fovea_rows = [&](int lr, int lc, uint32_t &mask) {
        mask = word_mask(4 * q, lc, lc + f_w);
        const int r_lo = lr - g * R;
        const int m_lo = max(r_lo, 0), m_hi = min(r_lo + f_h, R);
        return (mask && m_hi > m_lo) ? (((1u << m_hi) - 1u) & ~((1u << m_lo) - 1u)) : 0u;
    };
    // staged position (word index inside a buffer's fovea tile) of this thread's row r = 0
    auto fovea_pos = [&](int lr, int lc) { return (g * R - lr) * nw_max + (q - (lc >> 2)); };
    // prefetch of this group's plane for iteration j (env) into buffer j % NBUF
    auto prefetch = [&](int env, int j) {
        // buffer j % NBUF: its last tenant (iteration j - NBUF) was consumed before the group barrier that
        // ended iteration j - DIST - 1, which every thread of the group has passed
        const int b = j % NBUF;
        // s_loc entry j: its batch is published when the group first needs it, at the batch's first entry
        if ((j & 31) == 0) mbar_wait(&loc_full[(j / 32) % LOC_BATCHES], (j / 32 / LOC_BATCHES) & 1);
        const int4 lh = s_loc[j & (LOC_RING - 1)];
        int slot = lh.z + 1 + k;
        slot -= slot >= K ? K : 0;
        if (lead) {
            mbar_expect_tx(&full[k][b], PP * 4);
            bulk_g2s(bufs + b * buf_words, pcache + ((size_t)env * K + slot) * PP, PP * 4, &full[k][b]);
        }
        const uint32_t *plane = ring_w + ((size_t)env * K + slot) * PLANE_W;
        if constexpr (FS) {
            const int top = lh.x * Q, wb = top & ~3;  // ring word (inside a plane) the staging buffer starts at
            const int lw = lh.y >> 2, lastw = (lh.y + f_w - 1) >> 2;
#pragma unroll
            for (int a = 0; a < NJ; ++a) {
                if (ck_row[a] < 0) continue;
                const int rowbase = top + ck_row[a];
                const int cw = ((rowbase + lw) & ~3) + ck_c4[a];  // an aligned chunk that starts inside the plane ends inside it
                if (cw > rowbase + lastw) continue;
                cp_async16_s(bufs_s + (uint32_t)(b * buf_words + PP + (cw - wb)) * 4u, plane + cw);
            }
        } else if (active) {
            uint32_t mask;
            const uint32_t rows = fovea_rows(lh.x, lh.y, mask);
            if (rows) {
                const uint32_t *src = plane + word0;
                const uint32_t dst = bufs_s + (uint32_t)(b * buf_words + PP + fovea_pos(lh.x, lh.y)) * 4u;
                if (NW) {
                    prefetch_rows_imm<NW, 0>(rows, dst, src);
                } else {
#pragma unroll
                    for (int r = 0; r < R; ++r)
                        if (rows & (1u << r)) cp_async4_s(dst + (uint32_t)(r * nw_max) * 4u, src + r * Q);
                }
            }
        }
    };
    // W-expanded, biased squeezed row at float offset `so` of the staged squeeze
    auto t_row = [&](const float *sq, int so, uint64_t &t01, uint64_t &t23) {
        const float s0 = sq[so], s1 = sq[so + 1], s2 = sq[so + 2];
        const uint64_t p0 = pack2(s0, s0), p1 = pack2(s1, s1), p2 = pack2(s2, s2);
        t01 = ffma2(p2, wc01, ffma2(p1, wb01, ffma2(p0, wa01, bias2)));
        t23 = ffma2(p2, wc23, ffma2(p1, wb23, ffma2(p0, wa23, bias2)));
    };

    pdl_wait();       // ring, head, pcache, action, loc, out: not before the previous kernel in the stream has finished
    __syncthreads();  // mbarriers initialised
    if (tid < 32) loc_batch(0);
    {
        const int e0 = blockIdx.x;
#pragma unroll
        for (int j = 0; j < DIST; ++j) {
            if (e0 + j * G < N) prefetch(e0 + j * G, j);
            cp_async_commit();
        }
        if constexpr (FS) {   // the group's chunks of the first env, visible to the whole group after its barrier
            cp_async_wait<DIST - 1>();
            named_sync<GT>(1 + k);
        }
    }
    int it = 0;
    for (int e = blockIdx.x; e < N; e += G, ++it) {
        if (e + DIST * G < N) prefetch(e + DIST * G, it + DIST);
        cp_async_commit();
        if ((it & 31) == 0 && tid < 32) loc_batch(it + 32);
        const int b = it % NBUF;
        if constexpr (!FS) cp_async_wait<DIST>();    // this thread's own fovea words of env e
        mbar_wait(&full[k][b], (it / NBUF) & 1);     // the plane's cached squeeze (TMA)
        uint32_t *tile = tiles + (it & 1) * PLANE_W;
        if (active) {
            const int4 lh = s_loc[it & (LOC_RING - 1)];
            uint32_t fov_mask;
            const uint32_t rows = fovea_rows(lh.x, lh.y, fov_mask);
            const float *sq = bufs + b * buf_words;
            const uint32_t *sh = reinterpret_cast<const uint32_t *>(bufs + b * buf_words + PP) +
                                 (FS ? (int)word0 - ((lh.x * Q) & ~3) : fovea_pos(lh.x, lh.y));
            constexpr int SHP = FS ? Q : 0;   // staged words between two rows (FS: the ring's own pitch)
            uint32_t *o = tile + word0;
            uint64_t a0, a1, b0, b1, d0 = 0, d1 = 0;
            t_row(sq, so_t0, a0, a1);
            t_row(sq, so_mid + P, b0, b1);
            int t_have = 0;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int t = Gm::src(r) + 1;  // compile time: 0,0,1,1,1,1,2,...
                if (t != t_have) {              // resolved at compile time after unrolling
                    a0 = b0; a1 = b1;
                    t_row(sq, t + 1 == Gm::SPAN - 1 ? so_t6 : so_mid + (t + 1) * P, b0, b1);
                    t_have = t;
                }
                if (r == 0 || Gm::src(r) != Gm::src(r - 1)) { d0 = fsub2(a0, b0); d1 = fsub2(a1, b1); }
                // H weight of row r: the same for every segment (the plan checked it); at the clamped
                // border rows a == b, so the weight does not matter there
                const uint64_t w2 = pack2(ew.hw[r], ew.hw[r]);
                uint32_t u0, u1, u2, u3;
                unpack2(ffma2(w2, d0, b0), u0, u1);
                unpack2(ffma2(w2, d1, b1), u2, u3);
                uint32_t word = __byte_perm(__byte_perm(u0, u1, 0x0051), __byte_perm(u2, u3, 0x0051), 0x5410);
                if (rows & (1u << r))  // fovea rows: paste the sharp bytes (fov_env.py:385-386)
                    word = (word & ~fov_mask) | (sh[FS ? r * SHP : r * nw_max] & fov_mask);
                o[r * Q] = word;
            }
        }
        // the plane leaves as one TMA store; the store issued one iteration ago has finished reading this
        // iteration's tile's twin before anyone in the group writes it again (next iteration)
        fence_async_smem();
        if (lead) bulk_wait_read<0>();
        if constexpr (FS) cp_async_wait<DIST - 1>();   // this thread's chunks of the NEXT env, visible to the group after the barrier
        named_sync<GT>(1 + k);
        if (lead) {
            if ((it & 31) == 31) mbar_arrive(&loc_free[(it / 32) % LOC_BATCHES]);  // the group is done with this batch
            bulk_s2g(out + ((size_t)e * K + k) * (PLANE_W * 4), tile, PLANE_W * 4);
            bulk_commit();
        }
        if (p.norm_out) {   // uniform: the normalised copy of the same plane, 16 pixels per thread and pass; the tile is
                            // not written again before the group barrier of the NEXT iteration
            const uint4 *t4 = reinterpret_cast<const uint4 *>(tile);
            for (int i = lt; i < PLANE_W / 4; i += GT)
                norm_store16(p.norm_dt, t4[i], p.norm_out, ((size_t)e * K + k) * (PLANE_W / 4) + i);
        }
    }
    if (lead) bulk_wait_read<0>();  // shared memory must outlive the group's last store's reads
}


}  // namespace

// --------------------------------------------------------------------------- launchers
namespace {
// the normalised second output as a separate pass over the u8 output (kernels without the fused store)
cudaError_t normalize_after(cudaError_t e, const uint8_t *out, size_t bytes, void *norm_out, int norm_dt, cudaStream_t st) {
    if (e != cudaSuccess || !norm_out) return e;
    if (bytes % 16 != 0) return cudaErrorInvalidValue;   // the separate pass converts 16 pixels per thread
    return launch_normalize(out, bytes, norm_dt, norm_out, st);
}
}  // namespace

cudaError_t launch_observe_fixed(const DevPlan &p0, const uint8_t *ring, const int32_t *head, const double *action,
                                 const uint8_t *ctrl, int32_t *loc, int variant, uint8_t *out, void *norm_out, int norm_dt,
                                 cudaStream_t st) {
    DevPlan p = p0;
    p.norm_out = norm_out; p.norm_dt = norm_dt;
    const size_t out_bytes = (size_t)p.N * p.K * (variant == AGYM_OUT_CROP ? p.f_h * p.f_w : p.plane);
    cudaError_t e;
    const int crop_nwx = (p.f_w + 2) / 4 + 1;  // aligned words that cover f_w bytes at any byte offset
    const size_t crop_smem = a16((size_t)(p.K * p.f_h * p.f_w / 4) * 8) + (size_t)kCropWarps * p.K * p.f_h * crop_nwx * 4;
    CropV3Args c3;
    c3.nch = (p.f_w + 30) / 16;
    c3.g = p.f_w % 4 == 0 ? 1 : p.f_w % 2 == 0 ? 2 : 4;
    c3.gw = c3.g * p.f_w / 4;
    c3.ngroups = p.K * p.f_h / c3.g;
    c3.m_fh = 0xFFFFFFFFu / (uint32_t)p.f_h + 1u;
    c3.slice = (int)(16 + (size_t)p.K * p.f_h * c3.nch * 16);
    // RGB plans stage three times the planes per env (K = 9 at frame_stack 3: 8 envs x 21,076 B for f = 30 is past the
    // cap), so they run the same kernel with four envs per CTA (84,304 B); grey plans keep eight
    const int c3_warps = (p.C == 3 && (size_t)kCrop3Warps * (c3.slice + (size_t)p.K * p.f_h * p.f_w) > 100 * 1024) ? 4 : kCrop3Warps;
    const size_t crop3_smem = (size_t)c3_warps * (c3.slice + (size_t)p.K * p.f_h * p.f_w);
    if (variant == AGYM_OUT_CROP && (p.K * p.f_h * p.f_w) % 4 == 0 && (p.K * p.f_h) % c3.g == 0 && p.plane % 16 == 0 &&
        (reinterpret_cast<uintptr_t>(ring) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0 &&
        !g_disable_std && !g_crop_old && !g_crop_v2 && crop3_smem <= 100 * 1024) {
        const int grid = (p.N + c3_warps - 1) / c3_warps;
        // (plain launch: see launch_ingest_dmc about programmatic dependent launch and multi-wave grids)
#define AGYM_LAUNCH_CROP3(FW, W)                                                                                  \
    {                                                                                                             \
        if ((e = set_smem(k_observe_fixed_crop_v3<FW, W>, crop3_smem)) != cudaSuccess) return e;                   \
        k_observe_fixed_crop_v3<FW, W><<<grid, W * 32, crop3_smem, st>>>(p, ring, head, action, ctrl, loc, out, c3); \
    }
        if (c3_warps == 4) {
            if (p.f_w == 30) AGYM_LAUNCH_CROP3(30, 4)
            else AGYM_LAUNCH_CROP3(0, 4)
        } else if (p.f_w == 30) AGYM_LAUNCH_CROP3(30, kCrop3Warps)
        else AGYM_LAUNCH_CROP3(0, kCrop3Warps)
#undef AGYM_LAUNCH_CROP3
        return cudaGetLastError();   // the normalised output, if any, was written by the kernel
    }
    if (variant == AGYM_OUT_CROP && (p.K * p.f_h * p.f_w) % 4 == 0 && !g_disable_std && !g_crop_old &&
        crop_smem <= 64 * 1024 && p.K * p.f_h * crop_nwx * 4 + 4 < 65536) {
        if ((e = set_smem(k_observe_fixed_crop_v2, crop_smem)) != cudaSuccess) return e;
        // (plain launch: see launch_ingest_dmc about programmatic dependent launch and multi-wave grids)
        k_observe_fixed_crop_v2<<<(p.N + kCropWarps - 1) / kCropWarps, kCropWarps * 32, crop_smem, st>>>(p, ring, head, action, ctrl, loc, out, crop_nwx);
        return cudaGetLastError();   // the normalised output, if any, was written by the kernel
    } else if (variant == AGYM_OUT_CROP && (p.K * p.f_h * p.f_w) % 4 == 0 && !g_disable_std) {
        k_observe_fixed_crop_warp<<<(p.N + kThreads / 32 - 1) / (kThreads / 32), kThreads, 0, st>>>(p, ring, head, action, ctrl, loc, out);
    } else if (variant == AGYM_OUT_CROP) {
        k_observe_fixed<AGYM_OUT_CROP><<<p.N, kThreads, 0, st>>>(p, ring, head, action, ctrl, loc, out);
    } else if (variant == AGYM_OUT_MASK) {
        k_observe_fixed<AGYM_OUT_MASK><<<p.N, kThreads, 0, st>>>(p, ring, head, action, ctrl, loc, out);
    } else {
        const size_t smem = sizeof(float) * ((size_t)p.f_h * p.f_w + (size_t)p.f_h * p.S_w);
        if ((e = set_smem(k_observe_fixed<AGYM_OUT_RESIZE_FULL>, smem)) != cudaSuccess) return e;
        k_observe_fixed<AGYM_OUT_RESIZE_FULL><<<p.N, kThreads, smem, st>>>(p, ring, head, action, ctrl, loc, out);
    }
    return normalize_after(cudaGetLastError(), out, out_bytes, norm_out, norm_dt, st);
}

cudaError_t launch_observe_peripheral(const DevPlan &p0, const ExpandStd *ew, const uint8_t *ring, const int32_t *head,
                                      const float *pcache, const double *action, const uint8_t *ctrl, int32_t *loc,
                                      uint8_t *out, void *norm_out, int norm_dt, cudaStream_t st) {
    DevPlan p = p0;
    p.norm_out = norm_out; p.norm_dt = norm_dt;
    const size_t out_bytes = (size_t)p.N * p.K * p.plane;
    const size_t smem = a16(p.plane) + sizeof(float) * ((size_t)p.S_h * p.p_w + (size_t)p.p_h * p.p_w + (size_t)p.p_h * p.S_w);
    cudaError_t e;
    const int quads = p.S_w / 4;
    if (pcache && ew && ew->ok && (p.K == 4 || p.K == 3) && !g_disable_std && p.N < (1 << 30) &&
        (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(pcache) & 15) == 0) {  // TMA bulk copies
        const int nw_max = (p.f_w + 3) / 4 + 1;
        // per plane group: three input buffers { squeeze 400 f32 | staged fovea words } and two 1,764-word output tiles
        const size_t fov_words = ((size_t)p.f_h * nw_max + 3) & ~size_t(3);
        size_t fs = 4 * (size_t)p.K * (3 * (400 + fov_words) + 2 * 1764);
        // full-row staging (FS): 16-byte chunk copies; taken when two CTAs still fit an SM and two chunks per thread
        // suffice (21 * 4 * K rounded up to warps: at most 176 chunks per plane, within the 2 * 96 of a plane group)
        const size_t fs_rows = 4 * (size_t)p.K * (3 * (400 + (size_t)((p.f_h * 21 + 9) & ~3)) + 2 * 1764);
        const int std_threads = ((21 * 4 * p.K + 31) / 32) * 32;
        const bool full_rows = !g_std_nofs && fs_rows <= 112 * 1024 && p.K * p.f_h * ((p.f_w + 14) / 16 + 1) <= 2 * std_threads;
        int dev = 0, sms = 148, occ = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
#define AGYM_LAUNCH_STD(KK, NW, FSV)                                                                               \
    {                                                                                                              \
    if (fs <= 220 * 1024) {                                                                                        \
        const int threads = 96 * KK;   /* one 3-warp group per plane */                                            \
        if ((e = set_smem(k_observe_peripheral_std<KK, NW, FSV>, fs)) != cudaSuccess) return e;                    \
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_observe_peripheral_std<KK, NW, FSV>, threads, fs);   \
        if (occ >= 1) {                                                                                            \
            return launch_pdl(k_observe_peripheral_std<KK, NW, FSV>, dim3(std::min(p.N, sms * occ)), dim3(threads), fs, st, \
                              p, *ew, ring, head, pcache, action, ctrl, loc, out);                                 \
        }                                                                                                          \
    }                                                                                                              \
    }
        if (full_rows) {
            fs = fs_rows;
            if (p.K == 4) AGYM_LAUNCH_STD(4, 0, true)
            else AGYM_LAUNCH_STD(3, 0, true)
        }
        else if (p.K == 4 && nw_max == 9) AGYM_LAUNCH_STD(4, 9, false)
        else if (p.K == 4) AGYM_LAUNCH_STD(4, 0, false)
        else if (nw_max == 9) AGYM_LAUNCH_STD(3, 9, false)
        else AGYM_LAUNCH_STD(3, 0, false)
#undef AGYM_LAUNCH_STD
    }
    if (pcache && p.fast_expand && quads <= 64 && (p.p_h * p.p_w) % 4 == 0) {
        // rows per thread segment: a multiple of the expand pattern's period when S_h allows it
        // (84 -> 20 repeats every 21 rows), so the lanes of a warp switch source rows together
        int ysegs = std::max(1, 128 / quads);
        {
            int g = p.S_h, b2 = p.p_h;
            while (b2) { const int t = g % b2; g = b2; b2 = t; }   // gcd(S_h, p_h)
            const int period = p.S_h / g;
            while (ysegs > 1 && (p.S_h % ysegs != 0 || (p.S_h / ysegs) % period != 0)) --ysegs;
        }
        // phase B needs quads * ysegs threads, phase A at least one thread per column pair
        const int threads = ((std::max(quads * ysegs, 2 * quads) + 31) / 32) * 32;
        const int nw_max = (p.f_w + 3) / 4 + 1;
        const size_t buf_words = (((size_t)p.K * p.p_h * p.p_w + 3) & ~size_t(3)) + (((size_t)p.K * p.f_h * nw_max + 3) & ~size_t(3));
        const size_t fs = 4 * (2 * buf_words + (size_t)p.K * p.p_h * p.S_w) + 8 * ((size_t)p.S_h + 1);
        int dev = 0, sms = 148, occ = 1;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
#define AGYM_LAUNCH_PF(KG, PW)                                                                                     \
    {                                                                                                              \
        if ((e = set_smem(k_observe_peripheral_v2<KG, PW>, fs)) != cudaSuccess) return e;                          \
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_observe_peripheral_v2<KG, PW>, threads, fs);         \
        if (occ < 1) return cudaErrorInvalidConfiguration;                                                         \
        k_observe_peripheral_v2<KG, PW><<<std::min(p.N, sms * occ), threads, fs, st>>>(p, ring, head, pcache, action, \
                                                                                      ctrl, loc, out, ysegs);     \
    }
        if (p.K == 4 && p.plane == 7056) AGYM_LAUNCH_PF(4, 1764)
        else if (p.K == 3 && p.plane == 7056) AGYM_LAUNCH_PF(3, 1764)
        else if (p.C == 3 && p.K % 3 == 0 && p.plane == 7056) AGYM_LAUNCH_PF(3, 1764)   // RGB: 3 frames x 3 planes
        else if (p.K % 4 == 0) AGYM_LAUNCH_PF(4, 0)
        else if (p.K % 3 == 0) AGYM_LAUNCH_PF(3, 0)
        else if (p.K % 2 == 0) AGYM_LAUNCH_PF(2, 0)
        else AGYM_LAUNCH_PF(1, 0)
#undef AGYM_LAUNCH_PF
        return normalize_after(cudaGetLastError(), out, out_bytes, norm_out, norm_dt, st);
    }
    if (pcache) {
        if ((e = set_smem(k_observe_peripheral<true>, smem)) != cudaSuccess) return e;
        k_observe_peripheral<true><<<p.N, kThreads, smem, st>>>(p, ring, head, pcache, action, ctrl, loc, out);
    } else {
        if ((e = set_smem(k_observe_peripheral<false>, smem)) != cudaSuccess) return e;
        k_observe_peripheral<false><<<p.N, kThreads, smem, st>>>(p, ring, head, pcache, action, ctrl, loc, out);
    }
    return normalize_after(cudaGetLastError(), out, out_bytes, norm_out, norm_dt, st);
}


}  // namespace agym
