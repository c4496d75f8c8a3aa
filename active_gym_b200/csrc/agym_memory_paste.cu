// sm_100a kernel: foveal memory of the fixed fovea, pasted newest-on-top over a background
// (agym_observe_fixed_memory_paste).
#include "agym_device.cuh"

namespace agym {

namespace {

// The memory is agym_observe_fixed_memory's, byte for byte: per env a ring of up to 16 entries, each the packed
// (P, f_h, f_w) crop of one push padded to E = round_up(P f_h f_w, 16) bytes, plus its loc, plus {newest slot, held}.
// The observation differs: per plane, the background (zeros, or the periphery of the current ring) with the held
// windows written over it from the oldest to the newest, so at every pixel the newest window covering it wins.
//
// One CTA per env, plane by plane:
//   (i)   the tile (one S_h x S_w output plane in shared memory) starts as the background: zeros, or the expand of the
//         plane's cached squeeze, which arrives by one bulk copy issued while the previous plane finishes (BG_PERIPHERY);
//   (ii)  the older entries arrive oldest first by bulk copies (one per entry, plane and chunk of rows: the 16-byte hull
//         of the chunk's packed bytes) into the fixed ring of kPasteBufs shared-memory buffers on full mbarriers, issued
//         kPasteBufs units ahead across planes by thread 0 (k_observe_fixed_memory's pipeline); each entry row replaces
//         the tile bytes it covers by byte-masked word selects;
//   (iii) on a push the current window goes last, as ring words selected into the tile, and its bytes are packed into
//         the new entry's staging, which leaves by one bulk store per plane: the 16-byte-aligned range
//         [floor16(k A), floor16((k+1) A)) of the entry (A = f_h f_w); the <= 15 bytes past it are carried into the
//         next plane's store;
//   (iv)  the plane leaves as one TMA bulk store when d_out is 16-byte aligned, as 4-byte or byte stores otherwise
//         (uniform per launch); the normalised copy is written from the tile.
// Shared memory depends on the plan only, never on the depth.
constexpr int kPasteThreads = 128;
constexpr int kPasteBufs = 4;
constexpr int kPasteChunk = 2048;   // largest hull of one bulk copy of an older entry (rows of one plane)

constexpr int kBgZero = AGYM_BG_ZERO;
constexpr int kBgPeriphery = AGYM_BG_PERIPHERY;

struct PasteArgs {
    int M;            // depth
    int E;            // bytes per entry (multiple of 16)
    int rows;         // window rows per chunk
    int nchunk;       // chunks per plane
    int buf_stride;   // bytes per ring buffer: 16 spare + hull capacity + 16 spare
    int pk_bytes;     // staging of one plane of the new entry (+ carry and pad)
    int out_mode;     // 0: bulk store (16-byte aligned d_out), 1: 4-byte stores, 2: byte stores
    int sq_bulk;      // BG_PERIPHERY: the plane's squeeze arrives by one bulk copy (else by plain loads)
};

// Background of one column quad q over rows [y0, y1): Resize(S)(the cached squeeze sq [p_h][p_w]) from the plan's
// two-tap expand tables, in k_observe_peripheral_std's arithmetic (the restatement of agym_flexible.cu's periph_expand):
// W pass T = fma(w1, s[i0 + 1], fma(w0, s[i0], kBias)), H pass fma(w0, T[j] - T[j + 1], T[j + 1]), the pixel in byte 1
// of the float.  Bit-identical to that kernel's background at the standard geometry.
__device__ __forceinline__ void expand_quad(const DevPlan &p, const float *sq, int q, int y0, int y1, uint32_t *dst,
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
        if (j != j_have) {
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

template <int BG>
__global__ void __launch_bounds__(kPasteThreads) k_observe_memory_paste(const __grid_constant__ DevPlan p,
                                                                        const uint8_t *__restrict__ ring,
                                                                        const int32_t *__restrict__ head,
                                                                        const float *__restrict__ pcache,
                                                                        const double *__restrict__ action,
                                                                        const uint8_t *__restrict__ ctrl,
                                                                        int32_t *__restrict__ loc, uint8_t *__restrict__ mem,
                                                                        int32_t *__restrict__ mem_loc,
                                                                        int32_t *__restrict__ mem_state,
                                                                        uint8_t *__restrict__ out, const PasteArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ uint64_t s_full[kPasteBufs];
    __shared__ uint64_t s_sqbar;
    __shared__ int s_eloc[16][2];       // loc of the older entries, oldest first
    __shared__ int s_info[6];           // r0, c0, push, slot of the oldest older entry, their count, new slot
    __shared__ __align__(16) uint8_t s_carry[16];
    const int tid = threadIdx.x, n = blockIdx.x;
    const int P = p.K, fh = p.f_h, fw = p.f_w, A = fh * fw, M = a.M, Sw4 = p.S_w >> 2;
    uint8_t *s_tile = smem;                                       // [plane]
    uint8_t *s_pk = smem + align16((size_t)p.plane);              // [pk_bytes]
    uint8_t *s_buf = s_pk + a.pk_bytes;                           // [kPasteBufs][buf_stride]
    float *s_sq = reinterpret_cast<float *>(s_buf + kPasteBufs * a.buf_stride);   // BG_PERIPHERY: [p_h][p_w]
    float *s_t2 = s_sq + align16((size_t)p.p_h * p.p_w * 4) / 4;                  // generic expand: [p_h][S_w]
    uint32_t *tile32 = reinterpret_cast<uint32_t *>(s_tile);
    const int h = head[n];
    const int sq_floats = p.p_h * p.p_w;
    auto sq_src = [&](int k) {
        int slot = h + 1 + k;
        slot -= slot >= P ? P : 0;
        return pcache + ((size_t)n * P + slot) * sq_floats;
    };

    if (tid == 0) {
        for (int i = 0; i < kPasteBufs; ++i) mbar_init(&s_full[i], 1);
        mbar_init(&s_sqbar, 1);
        mbar_fence_init();
        if constexpr (BG == kBgPeriphery) {
            if (a.sq_bulk) {
                mbar_expect_tx(&s_sqbar, (uint32_t)(4 * sq_floats));
                bulk_g2s(s_sq, sq_src(0), (uint32_t)(4 * sq_floats), &s_sqbar);
            }
        }
        const LocIn li = load_loc_in(n, action, ctrl, loc);
        int r0, c0;
        apply_loc(p, li, r0, c0);
        loc[2 * n] = r0;
        loc[2 * n + 1] = c0;
        int newest = mem_state[2 * n], held = mem_state[2 * n + 1];
        newest = ((newest % M) + M) % M;           // a caller-written state stays inside the ring
        held = min(max(held, 0), M);
        if (li.mode == AGYM_FOV_RESET) held = 0;
        const bool push = li.mode != AGYM_FOV_KEEP;
        int last = newest, count = held;            // the newest older entry and the number of older entries
        if (push) {
            newest = held ? (newest + 1 == M ? 0 : newest + 1) : 0;
            held = min(held + 1, M);
            mem_loc[2 * ((size_t)n * M + newest)] = r0;
            mem_loc[2 * ((size_t)n * M + newest) + 1] = c0;
            last = newest == 0 ? M - 1 : newest - 1;
            count = held - 1;
        }
        mem_state[2 * n] = newest;
        mem_state[2 * n + 1] = held;
        int oldest = last - (count - 1);
        oldest += oldest < 0 ? M : 0;
        for (int j = 0, s = oldest; j < count; ++j, s = s + 1 == M ? 0 : s + 1) {
            // entries were written by this kernel; the clamp keeps a corrupted loc inside the tile
            s_eloc[j][0] = min(max(mem_loc[2 * ((size_t)n * M + s)], 0), p.S_h - fh);
            s_eloc[j][1] = min(max(mem_loc[2 * ((size_t)n * M + s) + 1], 0), p.S_w - fw);
        }
        s_info[0] = r0; s_info[1] = c0; s_info[2] = push; s_info[3] = oldest; s_info[4] = count; s_info[5] = newest;
    }
    __syncthreads();
    const int r0 = s_info[0], c0 = s_info[1], oldest = s_info[3], count = s_info[4], slot_new = s_info[5];
    const bool push = s_info[2] != 0;
    uint8_t *env_mem = mem + (size_t)n * M * a.E;
    const int per_plane = count * a.nchunk, units = P * per_plane;

    // unit u = (plane, older entry from the oldest, chunk of rows) -> its 16-byte hull into ring buffer u % kPasteBufs
    auto issue = [&](int u) {
        const int k = u / per_plane, rem = u - k * per_plane, j = rem / a.nchunk, c = rem - j * a.nchunk;
        int s = oldest + j;
        s -= s >= M ? M : 0;
        const int y0 = c * a.rows, y1 = min(y0 + a.rows, fh);
        const int lo = ((k * fh + y0) * fw) & ~15, hi = ((k * fh + y1) * fw + 15) & ~15;
        uint64_t *bar = &s_full[u % kPasteBufs];
        mbar_expect_tx(bar, (uint32_t)(hi - lo));
        bulk_g2s(s_buf + (u % kPasteBufs) * a.buf_stride + 16, env_mem + (size_t)s * a.E + lo, (uint32_t)(hi - lo), bar);
    };
    if (tid == 0)
        for (int u = 0; u < min(units, kPasteBufs); ++u) issue(u);

    const FastDiv fd_row(Sw4), fd_fw(fw);
    const int plane_words = p.plane >> 2;
    const int nw_win = ((c0 + fw - 1) >> 2) - (c0 >> 2) + 1;   // tile words a window row touches
    int u = 0;   // next unit to merge
    for (int k = 0; k < P; ++k) {
        if (tid == 0) bulk_wait_read<0>();   // the previous plane's stores have read the tile and the staging
        __syncthreads();
        // (i) the background
        if constexpr (BG == kBgPeriphery) {
            if (a.sq_bulk) {
                mbar_wait(&s_sqbar, (uint32_t)k & 1u);
            } else {
                const float *src = sq_src(k);
                for (int i = tid; i < sq_floats; i += kPasteThreads) s_sq[i] = __ldg(src + i);
                __syncthreads();
            }
            if (p.fast_expand) {
                const int nseg = min(p.S_h, max(1, kPasteThreads / Sw4)), rows = (p.S_h + nseg - 1) / nseg;
                for (int i = tid; i < Sw4 * nseg; i += kPasteThreads) {
                    const int g = i / Sw4, q = i - g * Sw4;
                    expand_quad(p, s_sq, q, g * rows, min(p.S_h, g * rows + rows), tile32 + g * rows * Sw4 + q, Sw4);
                }
            } else {   // the generic passes of k_observe_peripheral<true>: W pass into s_t2, H pass per word
                resample_w<float>(s_sq, p.p_w, s_t2, p.S_w, p.p_h, p.ex_w, tid, kPasteThreads);
                __syncthreads();
                for (int t = tid; t < plane_words; t += kPasteThreads) {
                    const int y = fd_row.div(t);
                    tile32[t] = resample_h_word(s_t2, p.S_w, p.ex_h, y, 4 * (t - y * Sw4));
                }
            }
        } else {
            for (int t = tid; t < plane_words; t += kPasteThreads) tile32[t] = 0u;
        }
        if (push) {
            const int base = (k * A) & ~15, carry = k * A - base;
            if (tid < carry) s_pk[tid] = s_carry[tid];
        }
        __syncthreads();
        if constexpr (BG == kBgPeriphery) {
            // the squeeze buffer is free: the next plane's squeeze arrives while this plane finishes
            if (tid == 0 && a.sq_bulk && k + 1 < P) {
                mbar_expect_tx(&s_sqbar, (uint32_t)(4 * sq_floats));
                bulk_g2s(s_sq, sq_src(k + 1), (uint32_t)(4 * sq_floats), &s_sqbar);
            }
        }
        // (ii) the older entries of this plane, oldest first
        for (int ue = u + per_plane; u < ue; ++u) {
            const int rem = u - k * per_plane, j = rem / a.nchunk, c = rem - j * a.nchunk;
            const int y0 = c * a.rows, y1 = min(y0 + a.rows, fh);
            const int lo = ((k * fh + y0) * fw) & ~15;
            const int er = s_eloc[j][0], ec = s_eloc[j][1];
            const int w0 = ec >> 2, nw = ((ec + fw - 1) >> 2) - w0 + 1;
            const uint8_t *buf = s_buf + (u % kPasteBufs) * a.buf_stride + 16;
            mbar_wait(&s_full[u % kPasteBufs], (uint32_t)(u / kPasteBufs) & 1u);
            const int items = (y1 - y0) * nw;
            for (int i = tid; i < items; i += kPasteThreads) {
                const int yy = i / nw, w = w0 + (i - yy * nw), y = y0 + yy;
                // byte of the buffer that lands in byte 0 of tile word w (>= -3: the 16 spare bytes in front)
                const int b = (k * fh + y) * fw - lo + 4 * w - ec;
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(buf + (b & ~3));
                const uint32_t m = word_mask(4 * w, ec, ec + fw);
                const uint32_t v = __funnelshift_r(wp[0], wp[1], (uint32_t)(b & 3) * 8u);
                uint32_t *t = tile32 + (er + y) * Sw4 + w;
                *t = (*t & ~m) | (v & m);
            }
            __syncthreads();   // buffer u % kPasteBufs is free, the entry's rows are written (the next entry overwrites them)
            if (tid == 0 && u + kPasteBufs < units) issue(u + kPasteBufs);
        }
        // (iii) the current window over everything, and its bytes packed into the new entry
        if (push) {
            int slot = h + 1 + k;
            slot -= slot >= P ? P : 0;
            const uint8_t *src = ring + ((size_t)n * P + slot) * p.plane;
            const uint32_t *src32 = reinterpret_cast<const uint32_t *>(src);
            for (int i = tid; i < fh * nw_win; i += kPasteThreads) {
                const int yy = i / nw_win, w = (c0 >> 2) + (i - yy * nw_win);
                const int t = (r0 + yy) * Sw4 + w;
                const uint32_t m = word_mask(4 * w, c0, c0 + fw);
                tile32[t] = (tile32[t] & ~m) | (__ldg(src32 + t) & m);
            }
            const int base = (k * A) & ~15, off = k * A - base;
            const int end = k + 1 == P ? a.E : (((k + 1) * A) & ~15);
            const int lim = k + 1 == P ? end - base : off + A;   // the last plane also zeroes the entry's pad bytes
            for (int i = tid; i < lim - off; i += kPasteThreads) {
                uint8_t v = 0;
                if (i < A) {
                    const int y = fd_fw.div(i), x = i - y * fw;
                    v = __ldg(src + (r0 + y) * p.S_w + c0 + x);
                }
                s_pk[off + i] = v;
            }
            fence_async_smem();
            __syncthreads();
            if (tid == 0 && end > base) bulk_s2g(env_mem + (size_t)slot_new * a.E + base, s_pk, (uint32_t)(end - base));
            // bytes past the store's end belong to the next plane's store
            if (k + 1 < P && tid < (k + 1) * A - end) s_carry[tid] = s_pk[end - base + tid];
        } else if (a.out_mode == 0) {
            fence_async_smem();
            __syncthreads();
        } else {
            __syncthreads();
        }
        // (iv) the finished plane
        uint8_t *dst = out + ((size_t)n * P + k) * p.plane;
        if (a.out_mode == 0) {
            if (tid == 0) bulk_s2g(dst, s_tile, (uint32_t)p.plane);
        } else if (a.out_mode == 1) {
            for (int t = tid; t < plane_words; t += kPasteThreads) reinterpret_cast<uint32_t *>(dst)[t] = tile32[t];
        } else {
            for (int t = tid; t < p.plane; t += kPasteThreads) dst[t] = s_tile[t];
        }
        if (tid == 0) bulk_commit();
        if (p.norm_out) {
            const uint4 *tv = reinterpret_cast<const uint4 *>(s_tile);
            const size_t v0 = ((size_t)n * P + k) * (p.plane >> 4);
            for (int t = tid; t < (p.plane >> 4); t += kPasteThreads) norm_store16(p.norm_dt, tv[t], p.norm_out, v0 + t);
        }
    }
    if (tid == 0) bulk_wait_read<0>();   // shared memory must outlive the stores' reads
}

}  // namespace

cudaError_t launch_observe_memory_paste(const DevPlan &p0, const uint8_t *ring, const int32_t *head, const float *pcache,
                                        const double *action, const uint8_t *ctrl, int32_t *loc, int depth, int background,
                                        uint8_t *mem, int32_t *mem_loc, int32_t *mem_state, uint8_t *out, void *norm_out,
                                        int norm_dt, cudaStream_t st) {
    DevPlan p = p0;
    p.norm_out = norm_out; p.norm_dt = norm_dt;
    const bool periph = background == AGYM_BG_PERIPHERY;
    PasteArgs a;
    a.M = depth;
    a.E = (int)memory_entry_bytes(p);
    a.rows = std::max(1, std::min(p.f_h, (kPasteChunk - 30) / p.f_w));
    a.nchunk = (p.f_h + a.rows - 1) / a.rows;
    a.buf_stride = (int)(16 + a16((size_t)a.rows * p.f_w + 30) + 16);
    a.pk_bytes = (int)a16((size_t)p.f_h * p.f_w + 32);
    const uintptr_t ob = reinterpret_cast<uintptr_t>(out);
    a.out_mode = (ob & 15) == 0 ? 0 : (ob & 3) == 0 ? 1 : 2;
    a.sq_bulk = periph && (p.p_h * p.p_w) % 4 == 0 && (reinterpret_cast<uintptr_t>(pcache) & 15) == 0;
    size_t smem = a16(p.plane) + (size_t)a.pk_bytes + (size_t)kPasteBufs * a.buf_stride;
    if (periph) smem += a16(4 * (size_t)p.p_h * p.p_w) + (p.fast_expand ? 0 : 4 * (size_t)p.p_h * p.S_w);
    cudaError_t e;
#define AGYM_LAUNCH_PASTE(BGV)                                                                                       \
    {                                                                                                                \
        if (!smem_fits(k_observe_memory_paste<BGV>, smem)) return cudaErrorNotSupported;                             \
        if ((e = set_smem(k_observe_memory_paste<BGV>, smem)) != cudaSuccess) return e;                              \
        k_observe_memory_paste<BGV><<<p.N, kPasteThreads, smem, st>>>(p, ring, head, pcache, action, ctrl, loc, mem, \
                                                                      mem_loc, mem_state, out, a);                   \
    }
    if (periph) AGYM_LAUNCH_PASTE(kBgPeriphery)
    else AGYM_LAUNCH_PASTE(kBgZero)
#undef AGYM_LAUNCH_PASTE
    return cudaGetLastError();
}

}  // namespace agym
