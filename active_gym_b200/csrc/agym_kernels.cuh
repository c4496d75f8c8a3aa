// Device-side parameter blocks and launcher prototypes shared by the kernel translation units agym_{ingest,observe,flexible,misc}.cu (device
// code + launchers) and agym_abi.cu (plan management + the extern "C" surface).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace agym {

// One antialiased-resample axis table inside the plan's device pool.
struct AxisRef {
    const int32_t *xmin;  // [n_out]
    const float *w;       // [n_out][taps]
    int32_t n_in, n_out, taps;
};

// Flexible fovea: per window size r (1..S) three tables per axis, stored as offsets (in
// 32-bit words) into the pool so one small index array serves every env.
struct FlexEntry {
    int32_t xmin_off, w_off, taps, n_out;
};

struct DevPlan {
    int32_t N, K, S_h, S_w, plane;      // plane = S_h * S_w; K = ring planes per env = frame_stack * C
    int32_t C;                          // planes per frame: 1 grey, 3 RGB (ring layout: include/agym_b200.h)
    int32_t raw_h, raw_w, raw_c;
    int32_t lw0, lw1, lw2;              // luma weights per channel position
    int32_t f_h, f_w, p_h, p_w;
    int32_t relative, init_r, init_c;
    double lo, hi;
    // cv2 bilinear raw -> obs (pool pointers)
    const int32_t *cx_s0, *cx_s1, *cx_coef;   // [S_w]
    const int32_t *cy_s0, *cy_s1, *cy_coef;   // [S_h]
    // antialiased axes (n_in -> n_out)
    AxisRef sq_w, sq_h;     // squeeze  S -> p      (fov_env.py:367)
    AxisRef ex_w, ex_h;     // expand   p -> S      (fov_env.py:368)
    AxisRef full_w, full_h; // resize_to_full f -> S (fov_env.py:120,182)
    // flexible fovea tables: index [axis][family][r], family 0 = r->f, 1 = f->r, 2 = r->S
    const FlexEntry *flex;  // [2][3][S_max+1]
    int32_t fov_tmax;       // widest r->f table (family 0) over both axes and every r
    // composed blur (Resize(f) then Resize(r)) per axis and window size r: [2][S_max+1]; blur_tmax = widest band
    const FlexEntry *flexb;
    int32_t blur_tmax;
    // W-axis blur operators in 16-bit fixed point: [S_max+1] {xmin_off, wq_off, halves of 8 taps, taps}; null = n/a
    const FlexEntry *flexq;
    // H-axis blur operators with duplicated weights {w, w}: [S_max+1] {xmin_off, w2_off, taps, n_out}
    const FlexEntry *flexh2;
    // {next env, CTAs done}: work counter of the persistent flexible kernel; zero between launches (the last CTA
    // re-arms it), so a plan must not run agym_observe_flexible on two streams at once
    int32_t *flex_counters;
    int32_t *err;           // per-launch: the caller's device error word (AGYM_ERR_RES_* bits) or null
    void *norm_out;         // per-launch: normalised second output (same shape as the u8 output) or null
    int32_t norm_dt;        // its element type, AGYM_DTYPE_*
    const int32_t *pool_i;  // pool base viewed as int32
    int32_t S_max;
    // ---- fast paths (0 = geometry not eligible, use the generic kernels)
    // ingest: per output-column pair {byte offset of the aligned word, PRMT selector, coef(x0), coef(x0+1)}
    // and per output row {b0 << 16, b1 << 16} (atari_env.py:74 fixed-point bilinear, dp2a form)
    int32_t fast_ingest;
    int32_t tma_span_rows[8];  // TMA ingest: largest source-row span of a unit when an env is cut into 1..8 units (0 = n/a)
    int32_t tma_period5;       // vertical scale 2.5: output row 2m samples raw rows {5m, 5m+1}, row 2m+1 {5m+3, 5m+4}
    int32_t std_gray;          // gray 210x160 -> 84x84 with the period-5 rows and (512,1536)/(1536,512) vertical weights: k_ingest_gray_std
    int32_t fast_ingest_rgb;   // 3-channel frames: every column pair's four source pixels lie among s0 .. s0 + 3
    const int4 *cx_pair;    // [S_w / 2]
    const int2 *cy_bs;      // [S_h]
    // squeeze along W from u8 rows: per output column {aligned byte offset, shift, first weight index}
    int32_t fast_squeeze, sqw_taps4;  // taps padded to a multiple of 4
    const int2 *sqw_ofs;    // [p_w] {aligned byte offset, 8 * (xmin & 3)}
    const float *sqw_w;     // [p_w][sqw_taps4]
    // the same pass in 16-bit fixed point (weights * 2^17, summing to 2^17 exactly) for IDP.2A: per output
    // column 8 words = 16 weights aligned to the 16-byte window at sqw_ofs.x (0 = geometry not eligible)
    int32_t squeeze_q;
    const uint32_t *sqw_q;  // [p_w][8]
    // expand p -> S as two taps: out = w0 * t[i0] + w1 * t[i0+1]  (w1 is given along W only)
    int32_t fast_expand;
    const int32_t *exw_i0, *exh_i0;   // [S_w], [S_h]
    const float *exw_w0, *exh_w0, *exw_w1;
};

// Host-side copy of the W-expand weights of the standard geometry (obs 84, periphery 20); passed
// to k_observe_peripheral_std by value so that they sit in the constant bank.  ok = the plan's
// tables follow the compile-time tap pattern of that kernel.
struct ExpandStd {
    float w0[84];   // W pass: out[x] = w0[x] * t[i0] + w1[x] * t[i0 + 1]
    float w1[84];
    float hw[21];   // H pass: weight of the upper row for row r of any 21-row segment
    int32_t ok;
};

cudaError_t launch_ingest_atari(const DevPlan &p, const uint8_t *fa, const uint8_t *fb, const uint8_t *flags,
                                uint8_t *ring, int32_t *head, float *pcache, cudaStream_t st);
// standard-geometry gray ingest (agym_ingest_std.cu); cudaErrorNotSupported = not eligible, use launch_ingest_atari's kernels
cudaError_t launch_ingest_gray_std(const DevPlan &p, const uint8_t *fa, const uint8_t *fb, const uint8_t *flags,
                                   uint8_t *ring, int32_t *head, float *pcache, cudaStream_t st);
cudaError_t launch_ingest_dmc(const DevPlan &p, const uint8_t *f, const uint8_t *flags, uint8_t *ring,
                              int32_t *head, float *pcache, cudaStream_t st);
cudaError_t launch_stack(const DevPlan &p, const uint8_t *ring, const int32_t *head, uint8_t *out, cudaStream_t st);
// norm_out / norm_dt: optional normalised second output of the observe launchers (null = none)
cudaError_t launch_observe_fixed(const DevPlan &p, const uint8_t *ring, const int32_t *head, const double *action,
                                 const uint8_t *ctrl, int32_t *loc, int variant, uint8_t *out, void *norm_out, int norm_dt,
                                 cudaStream_t st);
cudaError_t launch_observe_peripheral(const DevPlan &p, const ExpandStd *ew, const uint8_t *ring, const int32_t *head,
                                      const float *pcache, const double *action, const uint8_t *ctrl, int32_t *loc,
                                      uint8_t *out, void *norm_out, int norm_dt, cudaStream_t st);
// variant: AGYM_OUT_* or kOutPeriph; pcache: the squeeze cache kOutPeriph expands (null otherwise)
// cudaErrorNotSupported: no kernel fits the geometry (the generic kernel's two f32 planes exceed a block's shared memory)
constexpr int kOutPeriph = 4;   // flexible fovea over the peripheral background (agym_observe_flexible_peripheral)
cudaError_t launch_observe_flexible(const DevPlan &p, const uint8_t *ring, const int32_t *head, const float *pcache,
                                    const double *action, const int32_t *atype, const uint8_t *ctrl, int32_t *loc,
                                    int32_t *res, int variant, int pad_h, int pad_w, uint8_t *out, int32_t *err,
                                    void *norm_out, int norm_dt, cudaStream_t st);
// foveal memory of the fixed fovea (agym_memory.cu): bytes of one entry, and the observe launcher
size_t memory_entry_bytes(const DevPlan &p);
cudaError_t launch_observe_fixed_memory(const DevPlan &p, const uint8_t *ring, const int32_t *head, const double *action,
                                        const uint8_t *ctrl, int32_t *loc, int depth, uint8_t *mem, int32_t *mem_loc,
                                        int32_t *mem_state, uint8_t *out, void *norm_out, int norm_dt, cudaStream_t st);
// the same memory pasted newest-on-top over a background (agym_memory_paste.cu); background: AGYM_BG_*, pcache only for
// AGYM_BG_PERIPHERY; cudaErrorNotSupported: the plane and the periphery do not fit one block's shared memory
cudaError_t launch_observe_memory_paste(const DevPlan &p, const uint8_t *ring, const int32_t *head, const float *pcache,
                                        const double *action, const uint8_t *ctrl, int32_t *loc, int depth, int background,
                                        uint8_t *mem, int32_t *mem_loc, int32_t *mem_state, uint8_t *out, void *norm_out,
                                        int norm_dt, cudaStream_t st);
cudaError_t launch_normalize(const uint8_t *src, size_t n, int dtype, void *dst, cudaStream_t st);
cudaError_t launch_synth(uint8_t *dst, size_t n, uint64_t seed, cudaStream_t st);
cudaError_t launch_record_step(int n, int is_reset, const double *raw_reward, const uint8_t *done, const uint8_t *reset_mask,
                               int64_t *ep_len, double *cum_reward, const int32_t *loc, const int32_t *res,
                               int32_t *trace_row, cudaStream_t st);

}  // namespace agym
