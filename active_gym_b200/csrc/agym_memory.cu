// sm_100a kernel: foveal memory of the fixed fovea (agym_observe_fixed_memory).
#include "agym_device.cuh"

namespace agym {

namespace {

// The per-env memory is a ring of up to 16 entries, each the packed (P, f_h, f_w) crop of one push (the layout of
// agym_observe_fixed(AGYM_OUT_CROP)) padded to E = round_up(P f_h f_w, 16) bytes, plus its loc.  The observation is
// the pixelwise max of the entries held, each painted as its mask_out frame.
//
// One CTA per env, plane by plane:
//   (i)   the tile (one S_h x S_w output plane in shared memory) starts as this call's mask_out plane on a push — the
//         window's aligned ring words, the edge words masked, zero elsewhere (k_observe_fixed<AGYM_OUT_MASK>'s
//         arithmetic) — and as zeros on KEEP;
//   (ii)  on a push the window rows are packed from the tile into the new entry's bytes of this plane, which leave by one
//         cp.async.bulk store per plane: the store covers the 16-byte-aligned range [floor16(k A), floor16((k+1) A)) of
//         the entry (A = f_h f_w), and the <= 15 bytes past it are carried into the next plane's store;
//   (iii) the older entries arrive by bulk copies (one per entry, plane and chunk of rows: the 16-byte hull of the
//         chunk's packed bytes) into a fixed ring of kMemBufs shared-memory buffers on full mbarriers, issued kMemBufs
//         units ahead across planes by thread 0.  A chunk is at most kMemChunk bytes, so neither the depth nor the
//         fovea size sets the buffers' size;
//   (iv)  each entry row is merged with __vmaxu4 into the tile words it covers, from funnel-shifted buffer words whose
//         bytes outside the window are zero (zero is the identity of max: no read-modify-write masks on the tile);
//   (v)   the plane leaves as one TMA bulk store when d_out is 16-byte aligned, as 4-byte or byte stores otherwise
//         (uniform per launch); the normalised copy is written from the tile.
// The state update (RESET empties, APPLY / RESET push, KEEP pushes nothing) is thread 0's.
constexpr int kMemThreads = 128;
constexpr int kMemBufs = 4;
constexpr int kMemChunk = 2048;   // largest hull of one bulk copy of an older entry (rows of one plane)

struct MemArgs {
    int M;            // depth
    int E;            // bytes per entry (multiple of 16)
    int rows;         // window rows per chunk
    int nchunk;       // chunks per plane
    int buf_stride;   // bytes per ring buffer: 16 spare + hull capacity + 16 spare
    int pk_bytes;     // staging of one plane of the new entry (+ carry and pad)
    int out_mode;     // 0: bulk store (16-byte aligned d_out), 1: 4-byte stores, 2: byte stores
};

__global__ void __launch_bounds__(kMemThreads) k_observe_fixed_memory(const __grid_constant__ DevPlan p,
                                                                      const uint8_t *__restrict__ ring,
                                                                      const int32_t *__restrict__ head,
                                                                      const double *__restrict__ action,
                                                                      const uint8_t *__restrict__ ctrl,
                                                                      int32_t *__restrict__ loc, uint8_t *__restrict__ mem,
                                                                      int32_t *__restrict__ mem_loc,
                                                                      int32_t *__restrict__ mem_state, uint8_t *__restrict__ out,
                                                                      const MemArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    __shared__ uint64_t s_full[kMemBufs];
    __shared__ int s_eloc[16][2];       // loc of the older entries, newest first
    __shared__ int s_info[6];           // r0, c0, push, first slot of the older entries, their count, new slot
    __shared__ __align__(16) uint8_t s_carry[16];
    const int tid = threadIdx.x, n = blockIdx.x;
    const int P = p.K, fh = p.f_h, fw = p.f_w, A = fh * fw, M = a.M, Sw4 = p.S_w >> 2;
    uint8_t *s_tile = smem;                                       // [plane]
    uint8_t *s_pk = smem + align16((size_t)p.plane);              // [pk_bytes]
    uint8_t *s_buf = s_pk + a.pk_bytes;                           // [kMemBufs][buf_stride]
    uint32_t *tile32 = reinterpret_cast<uint32_t *>(s_tile);

    if (tid == 0) {
        for (int i = 0; i < kMemBufs; ++i) mbar_init(&s_full[i], 1);
        mbar_fence_init();
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
        int first = newest, count = held;
        if (push) {
            newest = held ? (newest + 1 == M ? 0 : newest + 1) : 0;
            held = min(held + 1, M);
            mem_loc[2 * ((size_t)n * M + newest)] = r0;
            mem_loc[2 * ((size_t)n * M + newest) + 1] = c0;
            first = newest == 0 ? M - 1 : newest - 1;
            count = held - 1;
        }
        mem_state[2 * n] = newest;
        mem_state[2 * n + 1] = held;
        for (int j = 0, s = first; j < count; ++j, s = s == 0 ? M - 1 : s - 1) {
            // entries were written by this kernel; the clamp keeps a corrupted loc inside the tile
            s_eloc[j][0] = min(max(mem_loc[2 * ((size_t)n * M + s)], 0), p.S_h - fh);
            s_eloc[j][1] = min(max(mem_loc[2 * ((size_t)n * M + s) + 1], 0), p.S_w - fw);
        }
        s_info[0] = r0; s_info[1] = c0; s_info[2] = push; s_info[3] = first; s_info[4] = count; s_info[5] = newest;
    }
    __syncthreads();
    const int r0 = s_info[0], c0 = s_info[1], first = s_info[3], count = s_info[4], slot_new = s_info[5];
    const bool push = s_info[2] != 0;
    const int h = head[n];
    uint8_t *env_mem = mem + (size_t)n * M * a.E;
    const int per_plane = count * a.nchunk, units = P * per_plane;

    // unit u = (plane, older entry, chunk of rows) -> its 16-byte hull into ring buffer u % kMemBufs
    auto issue = [&](int u) {
        const int k = u / per_plane, rem = u - k * per_plane, j = rem / a.nchunk, c = rem - j * a.nchunk;
        int s = first - j;
        s += s < 0 ? M : 0;
        const int y0 = c * a.rows, y1 = min(y0 + a.rows, fh);
        const int lo = ((k * fh + y0) * fw) & ~15, hi = ((k * fh + y1) * fw + 15) & ~15;
        uint64_t *bar = &s_full[u % kMemBufs];
        mbar_expect_tx(bar, (uint32_t)(hi - lo));
        bulk_g2s(s_buf + (u % kMemBufs) * a.buf_stride + 16, env_mem + (size_t)s * a.E + lo, (uint32_t)(hi - lo), bar);
    };
    if (tid == 0)
        for (int u = 0; u < min(units, kMemBufs); ++u) issue(u);

    const FastDiv fd_row(Sw4), fd_fw(fw);
    const int plane_words = p.plane >> 2;
    int u = 0;   // next unit to merge
    for (int k = 0; k < P; ++k) {
        if (tid == 0) bulk_wait_read<0>();   // the previous plane's stores have read the tile and the staging
        __syncthreads();
        // (i) the tile: this call's mask_out plane on a push, zeros on KEEP
        if (push) {
            int slot = h + 1 + k;
            slot -= slot >= P ? P : 0;
            const uint32_t *src = reinterpret_cast<const uint32_t *>(ring + ((size_t)n * P + slot) * p.plane);
            for (int t = tid; t < plane_words; t += kMemThreads) {
                const int y = fd_row.div(t), x0 = 4 * (t - y * Sw4);
                uint32_t m = 0u;
                if (y >= r0 && y < r0 + fh) m = word_mask(x0, c0, c0 + fw);
                tile32[t] = m ? (__ldg(src + t) & m) : 0u;
            }
            const int base = (k * A) & ~15, carry = k * A - base;
            if (tid < carry) s_pk[tid] = s_carry[tid];
        } else {
            for (int t = tid; t < plane_words; t += kMemThreads) tile32[t] = 0u;
        }
        __syncthreads();
        // (ii) the new entry's bytes of this plane, packed from the tile's window rows
        if (push) {
            const int base = (k * A) & ~15, off = k * A - base;
            const int end = k + 1 == P ? a.E : (((k + 1) * A) & ~15);
            const int lim = k + 1 == P ? end - base : off + A;   // the last plane also zeroes the entry's pad bytes
            for (int i = tid; i < lim - off; i += kMemThreads) {
                uint8_t v = 0;
                if (i < A) {
                    const int y = fd_fw.div(i), x = i - y * fw;
                    v = s_tile[(r0 + y) * p.S_w + c0 + x];
                }
                s_pk[off + i] = v;
            }
            fence_async_smem();
            __syncthreads();
            if (tid == 0 && end > base) {
                bulk_s2g(env_mem + (size_t)slot_new * a.E + base, s_pk, (uint32_t)(end - base));
                bulk_commit();
            }
            // bytes past the store's end belong to the next plane's store
            if (k + 1 < P && tid < (k + 1) * A - end) s_carry[tid] = s_pk[end - base + tid];
        }
        // (iii)+(iv) the older entries of this plane
        for (int ue = u + per_plane; u < ue; ++u) {
            const int rem = u - k * per_plane, j = rem / a.nchunk, c = rem - j * a.nchunk;
            const int y0 = c * a.rows, y1 = min(y0 + a.rows, fh);
            const int lo = ((k * fh + y0) * fw) & ~15;
            const int er = s_eloc[j][0], ec = s_eloc[j][1];
            const int w0 = ec >> 2, nw = ((ec + fw - 1) >> 2) - w0 + 1;
            const uint8_t *buf = s_buf + (u % kMemBufs) * a.buf_stride + 16;
            mbar_wait(&s_full[u % kMemBufs], (uint32_t)(u / kMemBufs) & 1u);
            const int items = (y1 - y0) * nw;
            for (int i = tid; i < items; i += kMemThreads) {
                const int yy = i / nw, w = w0 + (i - yy * nw), y = y0 + yy;
                // byte of the buffer that lands in byte 0 of tile word w (>= -3: the 16 spare bytes in front)
                const int b = (k * fh + y) * fw - lo + 4 * w - ec;
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(buf + (b & ~3));
                const uint32_t v = __funnelshift_r(wp[0], wp[1], (uint32_t)(b & 3) * 8u) & word_mask(4 * w, ec, ec + fw);
                uint32_t *t = tile32 + (er + y) * Sw4 + w;
                *t = __vmaxu4(*t, v);
            }
            __syncthreads();   // buffer u % kMemBufs is free, the tile rows are merged
            if (tid == 0 && u + kMemBufs < units) issue(u + kMemBufs);
        }
        // (v) the finished plane
        uint8_t *dst = out + ((size_t)n * P + k) * p.plane;
        if (a.out_mode == 0) {
            fence_async_smem();
            __syncthreads();
            if (tid == 0) {
                bulk_s2g(dst, s_tile, (uint32_t)p.plane);
                bulk_commit();
            }
        } else if (a.out_mode == 1) {
            for (int t = tid; t < plane_words; t += kMemThreads) reinterpret_cast<uint32_t *>(dst)[t] = tile32[t];
        } else {
            for (int t = tid; t < p.plane; t += kMemThreads) dst[t] = s_tile[t];
        }
        if (p.norm_out) {
            const uint4 *tv = reinterpret_cast<const uint4 *>(s_tile);
            const size_t v0 = ((size_t)n * P + k) * (p.plane >> 4);
            for (int t = tid; t < (p.plane >> 4); t += kMemThreads) norm_store16(p.norm_dt, tv[t], p.norm_out, v0 + t);
        }
    }
    if (tid == 0) bulk_wait_read<0>();   // shared memory must outlive the stores' reads
}

}  // namespace

size_t memory_entry_bytes(const DevPlan &p) { return ((size_t)p.K * p.f_h * p.f_w + 15) & ~size_t(15); }

cudaError_t launch_observe_fixed_memory(const DevPlan &p0, const uint8_t *ring, const int32_t *head, const double *action,
                                        const uint8_t *ctrl, int32_t *loc, int depth, uint8_t *mem, int32_t *mem_loc,
                                        int32_t *mem_state, uint8_t *out, void *norm_out, int norm_dt, cudaStream_t st) {
    DevPlan p = p0;
    p.norm_out = norm_out; p.norm_dt = norm_dt;
    MemArgs a;
    a.M = depth;
    a.E = (int)memory_entry_bytes(p);
    a.rows = std::max(1, std::min(p.f_h, (kMemChunk - 30) / p.f_w));
    a.nchunk = (p.f_h + a.rows - 1) / a.rows;
    a.buf_stride = (int)(16 + a16((size_t)a.rows * p.f_w + 30) + 16);
    a.pk_bytes = (int)a16((size_t)p.f_h * p.f_w + 32);
    const uintptr_t ob = reinterpret_cast<uintptr_t>(out);
    a.out_mode = (ob & 15) == 0 ? 0 : (ob & 3) == 0 ? 1 : 2;
    const size_t smem = a16(p.plane) + (size_t)a.pk_bytes + (size_t)kMemBufs * a.buf_stride;
    cudaError_t e;
    if ((e = set_smem(k_observe_fixed_memory, smem)) != cudaSuccess) return e;
    k_observe_fixed_memory<<<p.N, kMemThreads, smem, st>>>(p, ring, head, action, ctrl, loc, mem, mem_loc, mem_state, out, a);
    return cudaGetLastError();
}

}  // namespace agym
