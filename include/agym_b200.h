/*
 * agym_b200.h — C ABI of the B200-native active-perception observation path.
 *
 * This is the drop-in boundary for the observation code of elicassion/active-gym
 * (reference files cited as <file>:<lines> relative to /root/reference/active_gym/).
 * The reference has no FFI layer of its own (it is pure Python calling numpy / OpenCV /
 * torchvision per environment), so each entry point below names the reference METHOD it
 * replaces; INTEGRATION.md shows the ctypes stub a maintainer would put into those methods.
 *
 * Conventions
 *   - plain C, no torch / C++ types; every function returns 0 (AGYM_OK) or a negative
 *     agym_status, or a positive cudaError_t from the launch; nothing throws or exits.
 *   - the caller owns every buffer passed in.  `d_` parameters are DEVICE pointers on the current device,
 *     `h_` parameters are HOST pointers.  A plan owns only its small coefficient tables and a 16-byte work
 *     counter used by agym_observe_flexible (zero between launches); calls on one plan are stream-ordered:
 *     do not run the same plan's agym_observe_flexible on two streams at once (one plan per stream/shard).
 *   - all device work is enqueued on `stream` (a cudaStream_t passed as void*); no
 *     function synchronises unless its name ends in `_host`.
 *   - buffers should be 16-byte aligned (any cudaMalloc / torch allocation is): the TMA bulk-copy paths
 *     (cached squeeze in, observation tile out) need it; unaligned buffers are served by the slower
 *     table-driven kernels, never rejected.
 *   - u8 pixels everywhere: the reference's normalised float value is
 *     float64(float32(u)/255) for the u8 value u (SURVEY.md §8).
 *
 * Data layout in HBM (N = envs, K = frame_stack, C = obs_c planes per frame, P = K * C planes,
 * S = obs_size, f = fov_size)
 *   ring  u8  [N][P][S_h][S_w]  frame stack as a stack of P planes; head[n] is the plane index of the
 *                               NEWEST plane, logical order oldest->newest is (head+1)%P ... head.
 *                               Grey (C = 1): one plane per frame, head = slot of the newest frame.
 *                               RGB (C = 3): a frame occupies the C planes C*s .. C*s+C-1 of slot s (R, G, B),
 *                               and head = C*s + C-1 for the newest slot s; a push writes slot
 *                               s' = (head/C + 1) % K and sets head = (head + C) % P.  Read oldest->newest,
 *                               the planes are frame-major and channel-minor: the layout (K, C, S_h, S_w).
 *   head  i32 [N]
 *   loc   i32 [N][2]            (row, col) of the fovea's upper-left corner
 *   res   i32 [N][2]            (rows, cols) of the flexible fovea
 *   pcache f32 [N][P][p_h][p_w] optional cache of each ring plane's peripheral squeeze
 * Every observe call works plane by plane with one fov_loc / fov_res per env, so its outputs below are
 * written with P planes in place of K: (N, K, C, h, w) in memory.
 */
#ifndef AGYM_B200_H
#define AGYM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AGYM_ABI_VERSION 4

#if defined(__GNUC__)
#define AGYM_API __attribute__((visibility("default")))
#else
#define AGYM_API
#endif

typedef enum agym_status {
    AGYM_OK = 0,
    AGYM_ERR_INVALID_ARG = -1,   /* null pointer, non-positive size, fov >= obs ... */
    AGYM_ERR_UNSUPPORTED = -2,   /* geometry outside what the kernels are built for */
    AGYM_ERR_NO_DEVICE = -3,     /* no CUDA device / not an sm_100 part */
    AGYM_ERR_ALLOC = -4
} agym_status;

/* per-env ingest flags (u8) */
#define AGYM_FLAG_FRAME_A 1u     /* frame A is valid   (atari_env.py:125-126, t == 2)        */
#define AGYM_FLAG_FRAME_B 2u     /* frame B is valid   (atari_env.py:127-128, t == 3)        */
#define AGYM_FLAG_HARD_RESET 4u  /* zero-fill the stack first (atari_env.py:80-82,91)        */
#define AGYM_FLAG_IDLE 8u        /* env does not push a frame in this call                    */

/* per-env fovea control (u8), optional (NULL = AGYM_FOV_APPLY for every env) */
#define AGYM_FOV_APPLY 0u        /* apply the sensory action (fov_env.py:187-203)             */
#define AGYM_FOV_RESET 1u        /* loc = rint(fov_init_loc), res = fov_size (fov_env.py:149-150,250-251) */
#define AGYM_FOV_KEEP 2u         /* leave loc / res unchanged                                 */

/* output variants of the observe calls (fov_env.py:176-183, 289-296) */
#define AGYM_OUT_CROP 0          /* (K, f_h, f_w); flexible: padded (K, pad_h, pad_w)         */
#define AGYM_OUT_MASK 1          /* mask_out: (K, S_h, S_w), zero outside the fovea           */
#define AGYM_OUT_RESIZE_FULL 2   /* resize_to_full: (K, S_h, S_w)                             */
#define AGYM_OUT_RESIZE_FOV 3    /* flexible only: resize_to_fov, (K, f_h, f_w) = Resize(fov_size) of the unblurred window.
                                    Added without an ABI version bump (the struct and every signature are unchanged):
                                    a library that predates it rejects variant 3 with AGYM_ERR_INVALID_ARG */

/* bits of the device error word of agym_observe_flexible (d_err): FOV_RES actions the reference would fail on
 * (fov_env.py:322-324 stores the action unvalidated; the crop then raises for float bounds or a window larger than
 * the frame).  The kernels truncate and clamp to [1, S] and report it here instead. */
#define AGYM_ERR_RES_RANGE 1     /* a FOV_RES action outside [1, obs_size] (or NaN) was clamped   */
#define AGYM_ERR_RES_FRACTION 2  /* a FOV_RES action with a fractional part was truncated         */

/* element type of the normalised outputs (agym_normalize, d_out_norm of the observe calls) */
#define AGYM_DTYPE_F32 0
#define AGYM_DTYPE_F16 1
#define AGYM_DTYPE_BF16 2

/* sensory_action_type of the flexible fovea (fov_env.py:236-238) */
#define AGYM_ATYPE_FOV_LOC 0
#define AGYM_ATYPE_FOV_RES 1

/* Static configuration of one env batch: the fields of AtariEnvArgs / DMCEnvArgs that the
 * observation path reads (atari_env.py:25-39, dmc_env.py:56-76, fov_env.py:110-122,365). */
typedef struct agym_config {
    int32_t n_envs;              /* N                                                          */
    int32_t frame_stack;         /* K            (atari_env.py:55, dmc_env.py:90)              */
    int32_t obs_h, obs_w;        /* obs_size     (atari_env.py:59)                             */
    int32_t raw_h, raw_w, raw_c; /* simulator frame: Atari 210x160x{1 gray,3 RGB}; DMC obs x3  */
    int32_t luma_w[3];           /* 15-bit luma weight per channel position, when raw_c == 3   */
    int32_t fov_h, fov_w;        /* fov_size     (fov_env.py:110); 0 = no fovea (base env)     */
    int32_t periph_h, periph_w;  /* peripheral_res (fov_env.py:365); 0 = none                  */
    int32_t relative;            /* sensory_action_mode == "relative" (fov_env.py:114-118)     */
    double act_lo, act_hi;       /* sensory_action_space, relative mode (fov_env.py:116,170)   */
    double fov_init_loc[2];      /* fov_init_loc (fov_env.py:111,149-150)                      */
    int32_t no_antialias;        /* 0: torchvision Resize as installed today (antialias=True, fov_env.py:120,248,366-368);
                                    1: plain bilinear, the default of older torchvision releases on tensors     */
    int32_t obs_c;               /* planes per observed frame: 0 or 1 = grey (luma, dmc_env.py:182); 3 = RGB, the render's
                                    channels unconverted (DMC only: raw_c == 3 and raw == obs; dmc_env.py:122)         */
} agym_config;

typedef struct agym_plan agym_plan;   /* opaque: validated config + device coefficient tables */

AGYM_API int agym_abi_version(void);
AGYM_API const char *agym_status_string(int status);

/* Builds the coefficient tables on the host (OpenCV's 11-bit bilinear coefficients for
 * raw->obs, ATen's antialiased-bilinear weights for every resample the wrappers perform),
 * uploads them to the current device and returns a plan. */
AGYM_API int agym_plan_create(const agym_config *cfg, agym_plan **out_plan);
AGYM_API int agym_plan_destroy(agym_plan *plan);
/* sizes the caller needs to allocate (bytes) */
AGYM_API size_t agym_plan_ring_bytes(const agym_plan *plan);
AGYM_API size_t agym_plan_pcache_bytes(const agym_plan *plan);

/* Replaces AtariEnv._get_state + the frame logic of _step/_reset (atari_env.py:73-75,
 * 80-82, 91, 111-114, 121-133): per env gray(A),gray(B) -> cv2 INTER_LINEAR resize to
 * obs_size -> max -> push into the ring.  d_frames_a / d_frames_b: u8 [N][raw_h][raw_w][raw_c].
 * d_pcache (may be NULL): also refresh the pushed slot's peripheral squeeze cache.
 * Grey plans only (obs_c 0 / 1): AGYM_ERR_UNSUPPORTED on an RGB plan, as for the _packed variant. */
AGYM_API int agym_ingest_atari(const agym_plan *plan, const uint8_t *d_frames_a, const uint8_t *d_frames_b,
                      const uint8_t *d_flags, uint8_t *d_ring, int32_t *d_head, float *d_pcache,
                      void *stream);

/* Transport optimisation for host frame sources: cv2's bilinear resize reads only two raw rows per output
 * row (atari_env.py:74; 168 of 210 rows for 210 -> 84), so a frame may be shipped without the rows that are
 * never sampled.  agym_plan_used_rows returns their count and, if h_rows != NULL (capacity entries), the
 * ascending row indices; agym_ingest_atari_packed is agym_ingest_atari on frames laid out as
 * u8 [N][n_used_rows][raw_w][raw_c] holding exactly those rows.  Results are bit-identical. */
AGYM_API int agym_plan_used_rows(const agym_plan *plan, int32_t *h_rows, int32_t capacity);
AGYM_API int agym_ingest_atari_packed(const agym_plan *plan, const uint8_t *d_rows_a, const uint8_t *d_rows_b,
                             const uint8_t *d_flags, uint8_t *d_ring, int32_t *d_head, float *d_pcache,
                             void *stream);

/* Replaces DMCEnv._get_obs (pixel branch) + stack logic (dmc_env.py:175-183, 193-195,
 * 206-207, 228-230): luma of the rendered frame (grey plan) or its three channels as three planes
 * (RGB plan, see the ring layout) -> push.  d_frames: u8 [N][S_h][S_w][3].  A hard reset zeroes every
 * plane except the ones just pushed, and their cache entries. */
AGYM_API int agym_ingest_dmc(const agym_plan *plan, const uint8_t *d_frames, const uint8_t *d_flags,
                    uint8_t *d_ring, int32_t *d_head, float *d_pcache, void *stream);

/* Replaces np.stack(state_buffer) (atari_env.py:143, dmc_env.py:230): the base env's
 * observation, oldest -> newest.  d_out: u8 [N][K * C][S_h][S_w]. */
AGYM_API int agym_stack(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, uint8_t *d_out,
               void *stream);

/* Normalised second output of the three observe calls (SURVEY.md section 8f row 3): d_out_norm (may be NULL) receives,
 * in the layout of d_out, the value the reference hands to the agent — float32(u) / 255 (atari_env.py:75,
 * dmc_env.py:183) — as norm_dtype AGYM_DTYPE_F32 (bit-identical to the reference's float32) or rounded once more to
 * F16 / BF16.  The kernels of the standard geometries write it from the output tile they hold in shared memory / the
 * output words they hold in registers (no second pass over HBM); other geometries run agym_normalize on d_out behind
 * the observe kernel.  Both outputs must be 16-byte aligned and a multiple of 16 pixels long.
 *
 * Replaces FixedFovealEnv._fov_step + _get_fov_state (fov_env.py:166-203): updates d_loc
 * from the sensory action (f64 [N][2]; may be NULL when every env is RESET/KEEP) and writes
 * the observation.  d_out: u8 [N][K][f_h][f_w] (CROP) or [N][K][S_h][S_w] (MASK, RESIZE_FULL). */
AGYM_API int agym_observe_fixed(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
                       const double *d_action, const uint8_t *d_fov_ctrl, int32_t *d_loc,
                       int variant, uint8_t *d_out, void *d_out_norm, int norm_dtype, void *stream);

/* Replaces FixedFovealPeripheralEnv._get_fov_state (fov_env.py:375-388) with the loc update
 * fused in.  d_pcache may be NULL (the squeeze is then recomputed from the ring).
 * d_out: u8 [N][K][S_h][S_w]. */
AGYM_API int agym_observe_peripheral(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
                            const float *d_pcache, const double *d_action, const uint8_t *d_fov_ctrl,
                            int32_t *d_loc, uint8_t *d_out, void *d_out_norm, int norm_dtype, void *stream);

/* Replaces FlexibleFovealEnv._fov_step + _get_fov_state (fov_env.py:270-330).
 * d_atype: i32 [N] (NULL = all FOV_LOC).  CROP writes the variable-size patch into the
 * top-left corner of a zeroed [N][K][pad_h][pad_w] buffer (pad >= the largest res).
 * RESIZE_FOV writes the glimpse u8 [N][K][f_h][f_w]: each plane's unblurred window after this call's fovea update,
 * resampled to fov_size (torchvision Resize(fov_size), fov_env.py:248,284-285; the first half of the reference's blur),
 * within 0.5 LSB + 0.01 of the reference's float value (fp32 weights and accumulation on both axes); pad_h / pad_w are
 * ignored.  Any d_out alignment and any fov_size are served: the fast kernel when the tile K*f_h*f_w is a multiple of
 * 4 bytes and d_out is 4-byte aligned, the table-driven kernel otherwise.
 * Blurred pixels (res rows > fov rows) are within 0.5 LSB + 0.02 of the reference's float value: the W-axis
 * operator runs in 16-bit fixed point (<= 255 * taps / 2^17 LSB from the fp64 weights); windows that the
 * reference does not blur, the mask and the padding are bit exact.
 * d_err (may be NULL): one i32 the kernels OR the AGYM_ERR_RES_* bits into; the caller zeroes and reads it.
 * Size limit: a call the fast kernels cannot serve keeps two f32 planes (8 * S_h * S_w bytes) in the shared memory of
 * one block; past the device's limit (from about 172 x 172 observations on a B200) it returns AGYM_ERR_UNSUPPORTED
 * and launches nothing.  RESIZE_FULL always takes that kernel. */
AGYM_API int agym_observe_flexible(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
                          const double *d_action, const int32_t *d_atype, const uint8_t *d_fov_ctrl,
                          int32_t *d_loc, int32_t *d_res, int variant, int pad_h, int pad_w,
                          uint8_t *d_out, int32_t *d_err, void *d_out_norm, int norm_dtype, void *stream);

/* The flexible fovea over a peripheral background (a superset of the reference, which has no such wrapper):
 * FlexibleFovealEnv._fov_step (fov_env.py:300-330, with the same d_atype, d_fov_ctrl, d_res and d_err semantics as
 * agym_observe_flexible) followed by FixedFovealPeripheralEnv's observation (fov_env.py:366-368, 376, 385-386) with the
 * window pasted at its flexible size and place.  Per plane: bg = Resize(obs_size)(Resize(peripheral_res)(full)) from
 * the squeeze cache d_pcache (f32 [N][P][p_h][p_w], kept by the ingest calls; required); the window
 * full[r:r+rh, c:c+rw] is blurred by Resize(fov_res)(Resize(fov_size)(win)) iff rh > f_h (fov_env.py:276-280, 286-287)
 * and written over bg.  d_out: u8 [N][P][S_h][S_w], P = frame_stack * C.
 * Window pixels are bit for bit those of agym_observe_flexible(AGYM_OUT_MASK) on the same state (so bit exact when not
 * blurred, within 0.5 LSB + 0.02 of the reference's float value when blurred); background pixels are within 0.5 LSB +
 * 0.01 of it, and bit for bit agym_observe_peripheral's where that call runs its standard-geometry kernel (grey, 84x84
 * observations, 20x20 periphery).  Any d_out alignment is served (the fast kernel needs 16 bytes).
 * Size limit as for agym_observe_flexible, the table-driven kernel adding the background plane, the squeeze and its W
 * pass (S_h * S_w + 4 * p_h * (p_w + S_w) bytes): AGYM_ERR_UNSUPPORTED past it.
 * AGYM_ERR_INVALID_ARG for a plan without a fovea or a periphery and for NULL d_pcache or d_res.  Added without an ABI
 * version bump: the struct and every other signature are unchanged. */
AGYM_API int agym_observe_flexible_peripheral(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
                          const float *d_pcache, const double *d_action, const int32_t *d_atype,
                          const uint8_t *d_fov_ctrl, int32_t *d_loc, int32_t *d_res, uint8_t *d_out,
                          int32_t *d_err, void *d_out_norm, int norm_dtype, void *stream);

/* Foveal memory of the fixed fovea (a superset of the reference): the observation is the pixelwise max of the mask_out
 * observations of the env's last min(j, depth) pushes since its last fovea RESET, missing entries counting as zero
 * frames.  Per env and call, the fovea update of agym_observe_fixed runs first; then d_fov_ctrl decides: RESET empties the
 * memory and pushes, APPLY pushes, KEEP pushes nothing.  A push stores the (P, f_h, f_w) window after the update and its
 * loc, evicting the oldest entry once `depth` are held.  With no entry held the output is zero.  The memory follows the
 * fovea control only: an ingest AGYM_FLAG_HARD_RESET without a fovea RESET leaves it alone.
 *   d_mem       u8  [N][depth][E], E = round_up(P * f_h * f_w, 16): each entry the packed crop, in the layout
 *                   agym_observe_fixed(AGYM_OUT_CROP) writes.  Must be 16-byte aligned: the one buffer rejected for its
 *                   alignment (AGYM_ERR_INVALID_ARG), since the caller sizes it with agym_plan_memory_bytes.
 *   d_mem_loc   i32 [N][depth][2]: the loc of each entry.
 *   d_mem_state i32 [N][2]: {newest slot, entries held}; all zeros is an empty memory.
 * d_out: u8 [N][P][S_h][S_w] at any alignment.  AGYM_ERR_INVALID_ARG for depth outside 1..16, a NULL memory buffer and a
 * plan without a fovea.  Added without an ABI version bump: the struct and every other signature are unchanged. */
/* bytes of d_mem for a fovea memory of `depth` entries (1..16) for the plan's N envs (0 when invalid) */
AGYM_API size_t agym_plan_memory_bytes(const agym_plan *plan, int depth);
AGYM_API int agym_observe_fixed_memory(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
        const double *d_action, const uint8_t *d_fov_ctrl, int32_t *d_loc, int depth,
        uint8_t *d_mem, int32_t *d_mem_loc, int32_t *d_mem_state,
        uint8_t *d_out, void *d_out_norm, int norm_dtype, void *stream);

/* The same memory merged by pasting instead of by max (a superset of the reference): per plane, the background, then
 * the held windows written over it from the oldest to the newest, so at every pixel the newest window that covers it
 * wins.  With no entry held the output is the background alone.  The fovea update and the memory update (RESET empties
 * and pushes, APPLY pushes, KEEP pushes nothing) are agym_observe_fixed_memory's: d_mem, d_mem_loc and d_mem_state have
 * its layout and sizing (agym_plan_memory_bytes), and after the same sequence of calls hold the same bytes under either
 * merge.
 *   background AGYM_BG_ZERO: zeros; with depth 1 and every call pushing this is agym_observe_fixed(AGYM_OUT_MASK).
 *   background AGYM_BG_PERIPHERY: Resize(S)(Resize(p)(plane)) of the CURRENT ring (fov_env.py:366-368, 376), expanded
 *              from d_pcache; with depth 1 and every call pushing this is agym_observe_peripheral.  Its pixels are bit
 *              for bit agym_observe_peripheral's where that call runs its standard-geometry kernel (grey, 84x84, 20x20),
 *              and within 0.5 LSB + 0.01 of the reference's float value elsewhere.  Pasted pixels are exact.
 * d_pcache is ignored under AGYM_BG_ZERO.  d_out: u8 [N][P][S_h][S_w] at any alignment.  AGYM_ERR_INVALID_ARG for a
 * depth outside 1..16, a NULL memory buffer, a d_mem that is not 16-byte aligned, a plan without a fovea, an unknown
 * background, and AGYM_BG_PERIPHERY with a NULL d_pcache or a plan without a periphery.  AGYM_ERR_UNSUPPORTED when the
 * plane and the periphery do not fit one block's shared memory.  Added without an ABI version bump. */
#define AGYM_BG_ZERO 0        /* background of the pasted memory: zeros (mask_out)                 */
#define AGYM_BG_PERIPHERY 1   /* Resize(S)(Resize(p)(plane)) of the current ring, from d_pcache    */
AGYM_API int agym_observe_fixed_memory_paste(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head,
        const float *d_pcache, const double *d_action, const uint8_t *d_fov_ctrl, int32_t *d_loc, int depth,
        int background, uint8_t *d_mem, int32_t *d_mem_loc, int32_t *d_mem_state,
        uint8_t *d_out, void *d_out_norm, int norm_dtype, void *stream);

/* Replaces RecordWrapper's episode counters (fov_env.py:15-67) and the fov_loc / fov_res trace that
 * save_transition keeps when record=True (fov_env.py:152-154, 205-207, 253-256, 332-335), for N envs on the device.
 *   step  (is_reset = 0): ep_len += 1; cum_reward += d_raw_reward (f64 [N], info["raw_reward"]; NULL = 0)
 *   reset (is_reset = 1): both become 0 for the envs selected by d_reset_mask (u8 [N]; NULL = every env)
 *   d_ep_len i64 [N], d_cum_reward f64 [N]: the counters, updated in place (info["ep_len"], info["reward"])
 *   d_trace_row (may be NULL): i32 [N][6] = {fov_loc row, col, fov_res rows, cols, ep_len, valid} for this call;
 *     valid = 1 on a reset entry of a selected env and on a step whose d_done (u8 [N], NULL = none) is clear
 *     ("if not done: save_transition").  d_loc / d_res: i32 [N][2] or NULL (written as 0). */
AGYM_API int agym_record_step(int32_t n_envs, int is_reset, const double *d_raw_reward, const uint8_t *d_done,
                     const uint8_t *d_reset_mask, int64_t *d_ep_len, double *d_cum_reward, const int32_t *d_loc,
                     const int32_t *d_res, int32_t *d_trace_row, void *stream);

/* Host-only: the coefficient tables a plan would upload, for inspection and CPU-side tests.
 * agym_table_cv2: OpenCV INTER_LINEAR 11-bit coefficients of one axis (atari_env.py:74);
 * out arrays have n_dst entries, coef = c0 | (c1 << 16).
 * agym_table_aa: ATen antialiased-bilinear weights of one axis (fov_env.py:120,248,278,366-368);
 * h_xmin has n_out entries, h_w has n_out * (*taps) entries (capacity w_capacity floats). */
AGYM_API int agym_table_cv2(int n_src, int n_dst, int zero_frac_at_border, int32_t *h_s0, int32_t *h_s1, int32_t *h_coef);
AGYM_API int agym_table_aa(int n_in, int n_out, int antialias, int32_t *h_xmin, float *h_w, size_t w_capacity, int32_t *taps);
/* agym_table_blur: the flexible fovea's blur Resize(f) -> Resize(r) along one axis (fov_env.py:276-280) as ONE
 * banded r x r operator: h_xmin [r], h_w [r][*taps] float weights, and the 16-bit fixed-point form the W pass
 * of agym_observe_flexible multiplies with, h_q [r][*halves * 8] (weights * 2^16, every row sums to 2^16).
 * capacity: entries available in h_w and in h_q. */
AGYM_API int agym_table_blur(int r, int f, int antialias, int32_t *h_xmin, float *h_w, uint16_t *h_q, size_t capacity,
                             int32_t *taps, int32_t *halves);

/* Consumer-side convenience (SURVEY.md section 8f): u8 observations -> the reference's normalised value
 * float32(u) / 255 (atari_env.py:75, dmc_env.py:183) as a pass of its own.  AGYM_DTYPE_F32 is bit-identical to the
 * reference's float32; F16 / BF16 round that value once more.  n_bytes: number of pixels, a multiple of 16; both
 * pointers 16-byte aligned.  (The observe calls can write the same values as a second output, see above.) */
AGYM_API int agym_normalize(const uint8_t *d_src, size_t n_bytes, int dtype, void *d_dst, void *stream);

/* Benchmark / test helper: fills d_dst with a counter-based hash of (seed, byte index). */
AGYM_API int agym_synth_frames(uint8_t *d_dst, size_t n_bytes, uint64_t seed, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* AGYM_B200_H */
