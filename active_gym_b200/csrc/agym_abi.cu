// extern "C" surface of libagym_b200 (see include/agym_b200.h): plan management, argument
// validation and dispatch to the kernels.  No torch, no C++ types cross this boundary.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <vector>

#include "../../include/agym_b200.h"
#include "agym_kernels.cuh"
#include "agym_tables.h"

using namespace agym;

struct agym_plan {
    agym_config cfg;
    DevPlan dev;
    DevPlan dev_packed;             // same, for frames that carry only the raw rows the resize samples
    std::vector<int32_t> used_rows; // those rows, ascending (host)
    ExpandStd expand_std;  // host copy, see agym_kernels.cuh
    void *pool = nullptr;  // device: every coefficient table, one allocation
    size_t pool_bytes = 0;
    int device = -1;
};

namespace {

// Builder of the device pool: 32-bit words, every table 16-byte aligned.
struct Pool {
    std::vector<uint32_t> words;
    size_t add_i(const std::vector<int32_t> &v) {
        while (words.size() % 4) words.push_back(0);
        const size_t off = words.size();
        for (int32_t x : v) words.push_back(static_cast<uint32_t>(x));
        return off;
    }
    size_t add_f(const std::vector<float> &v) {
        while (words.size() % 4) words.push_back(0);
        const size_t off = words.size();
        for (float x : v) {
            uint32_t u;
            std::memcpy(&u, &x, 4);
            words.push_back(u);
        }
        return off;
    }
};

struct AxisOff {
    size_t xmin, w;
    int n_in, n_out, taps;
};

AxisOff add_axis(Pool &pool, int n_in, int n_out, bool aa) {
    const AaAxis ax = build_aa_axis(n_in, n_out, aa);
    return AxisOff{pool.add_i(ax.xmin), pool.add_f(ax.w), n_in, n_out, ax.taps};
}

AxisRef to_ref(const AxisOff &a, const uint32_t *base) {
    AxisRef r;
    r.xmin = reinterpret_cast<const int32_t *>(base + a.xmin);
    r.w = reinterpret_cast<const float *>(base + a.w);
    r.n_in = a.n_in; r.n_out = a.n_out; r.taps = a.taps;
    return r;
}

int validate(const agym_config &c) {
    if (c.n_envs <= 0 || c.frame_stack <= 0 || c.obs_h <= 0 || c.obs_w <= 0) return AGYM_ERR_INVALID_ARG;
    if (c.raw_h <= 0 || c.raw_w <= 0 || (c.raw_c != 1 && c.raw_c != 3)) return AGYM_ERR_INVALID_ARG;
    if (c.raw_c == 3) {  // 15-bit luma weights (cv2: 9798 / 19235 / 3735): the kernels evaluate them as 16-bit IDP.2A operands
        long sum = 0;
        for (int i = 0; i < 3; ++i) {
            if (c.luma_w[i] < 0 || c.luma_w[i] > 32767) return AGYM_ERR_INVALID_ARG;
            sum += c.luma_w[i];
        }
        if (sum > 32768) return AGYM_ERR_INVALID_ARG;
    }
    if (c.fov_h < 0 || c.fov_w < 0 || (c.fov_h == 0) != (c.fov_w == 0)) return AGYM_ERR_INVALID_ARG;
    if (c.periph_h < 0 || c.periph_w < 0 || (c.periph_h == 0) != (c.periph_w == 0)) return AGYM_ERR_INVALID_ARG;
    if (c.fov_h > 0) {
        // assert (fov_size < obs_size).all()  (fov_env.py:112)
        if (c.fov_h >= c.obs_h || c.fov_w >= c.obs_w) return AGYM_ERR_INVALID_ARG;
        // the reference does not clamp fov_init_loc (fov_env.py:149-150) and returns a short
        // crop when it is out of range; fixed-shape batched outputs cannot represent that
        const double r = std::nearbyint(c.fov_init_loc[0]), q = std::nearbyint(c.fov_init_loc[1]);
        if (!(r >= 0 && r <= c.obs_h - c.fov_h && q >= 0 && q <= c.obs_w - c.fov_w)) return AGYM_ERR_UNSUPPORTED;
        if (c.relative && !(c.act_lo <= c.act_hi)) return AGYM_ERR_INVALID_ARG;
    }
    if (c.periph_h > 0 && c.fov_h == 0) return AGYM_ERR_INVALID_ARG;
    // RGB observations: the render's channels as planes, so only DMC frames rendered at obs_size qualify
    if (c.obs_c != 0 && c.obs_c != 1 && c.obs_c != 3) return AGYM_ERR_INVALID_ARG;
    if (c.obs_c == 3 && (c.raw_c != 3 || c.raw_h != c.obs_h || c.raw_w != c.obs_w)) return AGYM_ERR_INVALID_ARG;
    // word/vector granularity the kernels are written for (84x84 obs, 210x160 raw satisfy all)
    if (c.obs_w % 4 != 0 || (c.obs_h * c.obs_w) % 16 != 0) return AGYM_ERR_UNSUPPORTED;
    if (c.obs_h > 255 || c.obs_w > 255 || c.raw_h > 4096 || c.raw_w > 4096) return AGYM_ERR_UNSUPPORTED;
    return AGYM_OK;
}

inline int planes_per_frame(const agym_config &c) { return c.obs_c == 3 ? 3 : 1; }
// ring planes per env: frame_stack * C
inline size_t ring_planes(const agym_config &c) { return static_cast<size_t>(c.frame_stack) * planes_per_frame(c); }

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }
inline int ret(cudaError_t e) { return e == cudaSuccess ? AGYM_OK : static_cast<int>(e); }

}  // namespace

extern "C" {

int agym_abi_version(void) { return AGYM_ABI_VERSION; }

const char *agym_status_string(int status) {
    switch (status) {
        case AGYM_OK: return "ok";
        case AGYM_ERR_INVALID_ARG: return "invalid argument";
        case AGYM_ERR_UNSUPPORTED: return "geometry not supported by the sm_100a kernels";
        case AGYM_ERR_NO_DEVICE: return "no usable CUDA device";
        case AGYM_ERR_ALLOC: return "allocation failed";
        default: return status > 0 ? cudaGetErrorString(static_cast<cudaError_t>(status)) : "unknown status";
    }
}

int agym_plan_create(const agym_config *cfg, agym_plan **out_plan) {
    if (!cfg || !out_plan) return AGYM_ERR_INVALID_ARG;
    *out_plan = nullptr;
    const int v = validate(*cfg);
    if (v != AGYM_OK) return v;
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess) return AGYM_ERR_NO_DEVICE;

    agym_plan *pl = new (std::nothrow) agym_plan();
    if (!pl) return AGYM_ERR_ALLOC;
    pl->cfg = *cfg;
    pl->device = dev;
    const agym_config &c = pl->cfg;

    const bool aa = c.no_antialias == 0;   // torchvision Resize: antialiased (today's default) or plain bilinear
    Pool pool;
    // cv2.resize raw -> obs (atari_env.py:74).  Unused by the DMC path (raw == obs).
    const Cv2Axis cx = build_cv2_axis(c.raw_w, c.obs_w, true), cy = build_cv2_axis(c.raw_h, c.obs_h, false);
    const size_t o_xs0 = pool.add_i(cx.s0), o_xs1 = pool.add_i(cx.s1), o_xcf = pool.add_i(cx.coef);
    const size_t o_ys0 = pool.add_i(cy.s0), o_ys1 = pool.add_i(cy.s1), o_ycf = pool.add_i(cy.coef);
    // packed frames: only the raw rows some output row samples, in ascending order (cv2 reads two of every
    // 2.5 rows for 210 -> 84, so a fifth of a frame never has to cross PCIe)
    std::vector<int32_t> used(cy.s0);
    used.insert(used.end(), cy.s1.begin(), cy.s1.end());
    std::sort(used.begin(), used.end());
    used.erase(std::unique(used.begin(), used.end()), used.end());
    std::vector<int32_t> ys0p(cy.s0.size()), ys1p(cy.s1.size());
    for (size_t y = 0; y < cy.s0.size(); ++y) {
        ys0p[y] = static_cast<int32_t>(std::lower_bound(used.begin(), used.end(), cy.s0[y]) - used.begin());
        ys1p[y] = static_cast<int32_t>(std::lower_bound(used.begin(), used.end(), cy.s1[y]) - used.begin());
    }
    const size_t o_ys0p = pool.add_i(ys0p), o_ys1p = pool.add_i(ys1p);
    pl->used_rows = used;
    AxisOff sq_w{}, sq_h{}, ex_w{}, ex_h{}, full_w{}, full_h{};
    if (c.periph_h > 0) {
        sq_w = add_axis(pool, c.obs_w, c.periph_w, aa); sq_h = add_axis(pool, c.obs_h, c.periph_h, aa);
        ex_w = add_axis(pool, c.periph_w, c.obs_w, aa); ex_h = add_axis(pool, c.periph_h, c.obs_h, aa);
    }
    const int s_max = c.obs_h > c.obs_w ? c.obs_h : c.obs_w;
    size_t o_flex = 0, o_flexb = 0, o_flexq = 0, o_flexh2 = 0, o_counters = 0;
    bool have_flexq = false;
    int blur_tmax = 0, fov_tmax = 0;
    if (c.fov_h > 0) {
        full_w = add_axis(pool, c.fov_w, c.obs_w, aa); full_h = add_axis(pool, c.fov_h, c.obs_h, aa);
        // flexible fovea: for every window size r, r->f, f->r and r->S on both axes
        std::vector<int32_t> index(static_cast<size_t>(2) * 3 * (s_max + 1) * 4, 0);
        for (int axis = 0; axis < 2; ++axis) {
            const int f = axis == 0 ? c.fov_h : c.fov_w, S = axis == 0 ? c.obs_h : c.obs_w;
            for (int fam = 0; fam < 3; ++fam)
                for (int r = 1; r <= S; ++r) {
                    const int n_in = fam == 1 ? f : r, n_out = fam == 0 ? f : (fam == 1 ? r : S);
                    const AxisOff a = add_axis(pool, n_in, n_out, aa);
                    int32_t *e = index.data() + (static_cast<size_t>(axis * 3 + fam) * (s_max + 1) + r) * 4;
                    e[0] = static_cast<int32_t>(a.xmin); e[1] = static_cast<int32_t>(a.w); e[2] = a.taps; e[3] = a.n_out;
                    if (fam == 0) fov_tmax = std::max(fov_tmax, a.taps);
                }
        }
        o_flex = pool.add_i(index);
        // composed blur operators of the flexible fovea, one per axis and window size
        std::vector<int32_t> bindex(static_cast<size_t>(2) * (s_max + 1) * 4, 0);
        for (int axis = 0; axis < 2; ++axis) {
            const int f = axis == 0 ? c.fov_h : c.fov_w, S = axis == 0 ? c.obs_h : c.obs_w;
            for (int r = 1; r <= S; ++r) {
                const AaAxis ax = build_blur_axis(r, f, aa);
                int32_t *e = bindex.data() + (static_cast<size_t>(axis) * (s_max + 1) + r) * 4;
                e[0] = static_cast<int32_t>(pool.add_i(ax.xmin)); e[1] = static_cast<int32_t>(pool.add_f(ax.w));
                e[2] = ax.taps; e[3] = ax.n_out;
                blur_tmax = std::max(blur_tmax, ax.taps);
            }
        }
        o_flexb = pool.add_i(bindex);
        // the W-axis operators once more in 16-bit fixed point for IDP.2A (k_observe_flexible_v3): per output
        // column 8 weights per half (taps 0-7, 8-15) starting at xmin, scaled by 2^16 and rounded by largest
        // remainder so that a row sums to 2^16 exactly (a lone weight of 1.0 is stored as 65535)
        if (blur_tmax <= 16) {
            std::vector<int32_t> qindex(static_cast<size_t>(s_max + 1) * 4, 0);
            for (int r = 1; r <= c.obs_w; ++r) {
                const AaAxis ax = build_blur_axis(r, c.fov_w, aa);
                int nh = 1;
                const std::vector<uint32_t> qu = quantize_axis_q16(ax, &nh);
                const std::vector<int32_t> q(qu.begin(), qu.end());
                int32_t *e = qindex.data() + static_cast<size_t>(r) * 4;
                e[0] = static_cast<int32_t>(pool.add_i(ax.xmin)); e[1] = static_cast<int32_t>(pool.add_i(q));
                e[2] = nh; e[3] = ax.taps;
            }
            o_flexq = pool.add_i(qindex);
            // H-axis operators with every weight stored twice ({w, w} is the FFMA2 operand), padded to 16 bytes
            std::vector<int32_t> hindex(static_cast<size_t>(s_max + 1) * 4, 0);
            for (int r = 1; r <= c.obs_h; ++r) {
                const AaAxis ax = build_blur_axis(r, c.fov_h, aa);
                std::vector<float> w2;
                for (float w : ax.w) { w2.push_back(w); w2.push_back(w); }
                while (w2.size() % 4) w2.push_back(0.f);
                int32_t *e = hindex.data() + static_cast<size_t>(r) * 4;
                e[0] = static_cast<int32_t>(pool.add_i(ax.xmin)); e[1] = static_cast<int32_t>(pool.add_f(w2));
                e[2] = ax.taps; e[3] = ax.n_out;
            }
            o_flexh2 = pool.add_i(hindex);
            o_counters = pool.add_i(std::vector<int32_t>(4, 0));
            have_flexq = true;
        }
    }

    // ---- fast-path tables (see DevPlan)
    // ingest: dp2a form of the horizontal pass, two output columns per thread
    bool fast_ingest = (c.obs_w % 2 == 0) && (c.obs_w / 2 <= 256);
    std::vector<int32_t> pair_tab, ybs_tab;
    bool fast_ingest_rgb = true;
    for (int x0 = 0; fast_ingest && x0 < c.obs_w; x0 += 2) {
        const int s[4] = {cx.s0[x0], cx.s1[x0], cx.s0[x0 + 1], cx.s1[x0 + 1]};
        const int base = s[0] & ~3;
        int sel = 0;
        for (int k = 0; k < 4; ++k) {
            const int o = s[k] - base;
            if (o < 0 || o > 7) fast_ingest = false;
            sel |= (o & 7) << (4 * k);
        }
        pair_tab.insert(pair_tab.end(), {base, sel, cx.coef[x0], cx.coef[x0 + 1]});
        for (int k = 0; k < 4; ++k) fast_ingest_rgb = fast_ingest_rgb && s[k] - s[0] >= 0 && s[k] - s[0] <= 3;
    }
    for (int y = 0; y < c.obs_h; ++y) {
        ybs_tab.push_back((cy.coef[y] & 0xffff) << 16);
        ybs_tab.push_back((cy.coef[y] >> 16) << 16);
    }
    size_t o_pair = 0, o_ybs = 0;
    if (fast_ingest) { o_pair = pool.add_i(pair_tab); o_ybs = pool.add_i(ybs_tab); }
    // squeeze along W straight from u8 rows: a 16-byte window per output column
    bool fast_squeeze = c.periph_h > 0;
    size_t o_sqofs = 0, o_sqw = 0, o_sqq = 0;
    bool squeeze_q = false;
    int sq_taps4 = 0;
    if (fast_squeeze) {
        const AaAxis ax = build_aa_axis(c.obs_w, c.periph_w, aa);
        sq_taps4 = (ax.taps + 3) & ~3;
        std::vector<int32_t> ofs;
        std::vector<float> wts(static_cast<size_t>(ax.n_out) * sq_taps4, 0.f);
        for (int i = 0; i < ax.n_out; ++i) {
            if ((ax.xmin[i] & 3) + ax.taps > 16) fast_squeeze = false;
            ofs.push_back(ax.xmin[i] & ~3);
            ofs.push_back(8 * (ax.xmin[i] & 3));
            for (int j = 0; j < ax.taps; ++j) wts[static_cast<size_t>(i) * sq_taps4 + j] = ax.w[static_cast<size_t>(i) * ax.taps + j];
        }
        if (fast_squeeze) { o_sqofs = pool.add_i(ofs); o_sqw = pool.add_f(wts); }
        // fixed-point form: q_j = round(w_j * 2^17), largest weight adjusted so that the sum is 2^17 exactly
        squeeze_q = fast_squeeze;
        std::vector<int32_t> qtab(static_cast<size_t>(ax.n_out) * 8, 0);
        for (int i = 0; squeeze_q && i < ax.n_out; ++i) {
            std::vector<long> q(ax.taps);
            long sum = 0;
            int jmax = 0;
            for (int j = 0; j < ax.taps; ++j) {
                q[j] = std::lround(static_cast<double>(ax.w[static_cast<size_t>(i) * ax.taps + j]) * 131072.0);
                sum += q[j];
                if (q[j] > q[jmax]) jmax = j;
            }
            q[jmax] += 131072 - sum;
            for (int j = 0; j < ax.taps; ++j) {
                if (q[j] < 0 || q[j] > 32767) squeeze_q = false;
                const int t = (ax.xmin[i] & 3) + j;  // position inside the aligned 16-byte window
                qtab[static_cast<size_t>(i) * 8 + t / 2] |= static_cast<int32_t>(static_cast<uint32_t>(q[j] & 0xffff) << (16 * (t & 1)));
            }
        }
        if (squeeze_q) o_sqq = pool.add_i(qtab);
    }
    // expand p -> S as two-tap lerps (plain bilinear upsampling: antialiasing is inactive)
    bool fast_expand = c.periph_h > 0 && c.periph_h < c.obs_h && c.periph_w < c.obs_w && c.periph_h >= 2 && c.periph_w >= 2;
    size_t o_ewi = 0, o_eww = 0, o_ehi = 0, o_ehw = 0, o_eww1 = 0;
    if (fast_expand) {
        auto lerp = [&](int n_in, int n_out, std::vector<int32_t> &i0, std::vector<float> &w0, std::vector<float> &w1) {
            const AaAxis ax = build_aa_axis(n_in, n_out, aa);
            for (int i = 0; i < n_out; ++i) {
                int first = -1, last = -1;
                for (int j = 0; j < ax.taps; ++j)
                    if (ax.w[static_cast<size_t>(i) * ax.taps + j] != 0.f) { if (first < 0) first = j; last = j; }
                if (first < 0 || last - first > 1) { fast_expand = false; return; }
                const int a = ax.xmin[i] + first;
                if (last > first) {
                    i0.push_back(a);
                    w0.push_back(ax.w[static_cast<size_t>(i) * ax.taps + first]);
                    w1.push_back(ax.w[static_cast<size_t>(i) * ax.taps + last]);
                }
                else if (a + 1 <= n_in - 1) { i0.push_back(a); w0.push_back(1.f); w1.push_back(0.f); }
                else { i0.push_back(a - 1); w0.push_back(0.f); w1.push_back(1.f); }
            }
        };
        std::vector<int32_t> wi, hi;
        std::vector<float> ww, hw, ww1, hw1;
        lerp(c.periph_w, c.obs_w, wi, ww, ww1);
        if (fast_expand) lerp(c.periph_h, c.obs_h, hi, hw, hw1);
        if (fast_expand) {
            o_ewi = pool.add_i(wi); o_eww = pool.add_f(ww); o_eww1 = pool.add_f(ww1);
            o_ehi = pool.add_i(hi); o_ehw = pool.add_f(hw);
            // standard geometry: do the tables follow k_observe_peripheral_std's compile-time pattern,
            // i0 = clamp(floor((40 i - 64) / 168), 0, 18) with single-tap borders on both axes?
            ExpandStd &es = pl->expand_std;
            bool ok = c.obs_h == 84 && c.obs_w == 84 && c.periph_h == 20 && c.periph_w == 20;
            for (int i = 0; ok && i < 84; ++i) {
                const int raw = (40 * i - 64 + 168 * 4) / 168 - 4;
                const int want = raw < 0 ? 0 : (raw > 18 ? 18 : raw);
                ok = wi[i] == want && hi[i] == want;
                if (raw < 0) ok = ok && ww[i] == 1.f && hw[i] == 1.f;       // out = t[0]
                if (raw > 18) ok = ok && ww[i] == 0.f && hw[i] == 0.f;      // out = t[19]
            }
            // H weights repeat every 21 rows bit for bit, except at the clamped border rows (0, 1, 82, 83)
            // where both taps read the same squeezed row and the weight is irrelevant
            for (int i = 2; ok && i < 82; ++i) ok = std::memcmp(&hw[i], &hw[21 + (i % 21)], sizeof(float)) == 0 || (21 + i % 21 >= 82);
            if (ok) {
                for (int i = 0; i < 84; ++i) { es.w0[i] = ww[i]; es.w1[i] = ww1[i]; }
                for (int r = 0; r < 21; ++r) es.hw[r] = hw[21 + r];
            }
            es.ok = ok;
        }
    }

    pl->pool_bytes = pool.words.size() * 4;
    if (cudaMalloc(&pl->pool, pl->pool_bytes) != cudaSuccess) { delete pl; return AGYM_ERR_ALLOC; }
    const cudaError_t e = cudaMemcpy(pl->pool, pool.words.data(), pl->pool_bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(pl->pool); delete pl; return static_cast<int>(e); }

    const uint32_t *base = static_cast<const uint32_t *>(pl->pool);
    DevPlan &d = pl->dev;
    std::memset(&d, 0, sizeof(d));
    d.N = c.n_envs; d.C = planes_per_frame(c); d.K = c.frame_stack * d.C; d.S_h = c.obs_h; d.S_w = c.obs_w; d.plane = c.obs_h * c.obs_w;
    d.raw_h = c.raw_h; d.raw_w = c.raw_w; d.raw_c = c.raw_c;
    d.lw0 = c.luma_w[0]; d.lw1 = c.luma_w[1]; d.lw2 = c.luma_w[2];
    d.f_h = c.fov_h; d.f_w = c.fov_w; d.p_h = c.periph_h; d.p_w = c.periph_w;
    d.relative = c.relative;
    d.init_r = static_cast<int32_t>(std::nearbyint(c.fov_init_loc[0]));
    d.init_c = static_cast<int32_t>(std::nearbyint(c.fov_init_loc[1]));
    d.lo = c.act_lo; d.hi = c.act_hi;
    auto ip = [&](size_t off) { return reinterpret_cast<const int32_t *>(base + off); };
    d.cx_s0 = ip(o_xs0); d.cx_s1 = ip(o_xs1); d.cx_coef = ip(o_xcf);
    d.cy_s0 = ip(o_ys0); d.cy_s1 = ip(o_ys1); d.cy_coef = ip(o_ycf);
    if (c.periph_h > 0) {
        d.sq_w = to_ref(sq_w, base); d.sq_h = to_ref(sq_h, base);
        d.ex_w = to_ref(ex_w, base); d.ex_h = to_ref(ex_h, base);
    }
    if (c.fov_h > 0) {
        d.full_w = to_ref(full_w, base); d.full_h = to_ref(full_h, base);
        d.flex = reinterpret_cast<const FlexEntry *>(base + o_flex);
        d.flexb = reinterpret_cast<const FlexEntry *>(base + o_flexb);
        d.blur_tmax = blur_tmax;
        d.fov_tmax = fov_tmax;
        d.flexq = have_flexq ? reinterpret_cast<const FlexEntry *>(base + o_flexq) : nullptr;
        d.flexh2 = have_flexq ? reinterpret_cast<const FlexEntry *>(base + o_flexh2) : nullptr;
        d.flex_counters = have_flexq ? reinterpret_cast<int32_t *>(static_cast<uint32_t *>(pl->pool) + o_counters) : nullptr;
    }
    d.pool_i = reinterpret_cast<const int32_t *>(base);
    d.S_max = s_max;
    d.fast_ingest = fast_ingest;
    d.fast_ingest_rgb = fast_ingest && fast_ingest_rgb && c.raw_c == 3;
    auto spans = [&](const std::vector<int32_t> &s0, const std::vector<int32_t> &s1, int32_t *out4) {
        for (int u = 1; u <= 8; ++u) {  // row span of the largest unit when the output rows are cut into u units
            out4[u - 1] = 0;
            if (c.obs_h % u != 0) continue;
            const int R = c.obs_h / u;
            int span = 0;
            bool monotone = true;
            for (int k = 0; k < u; ++k) {
                const int lo = s0[k * R], hi = s1[k * R + R - 1];
                for (int y = k * R; y < k * R + R; ++y) monotone = monotone && s0[y] >= lo && s1[y] <= hi;
                span = std::max(span, hi - lo + 1);
            }
            // a stage holds both frames' spans; keep two stages well inside one SM's shared memory
            if (monotone && 2 * (2 * (static_cast<size_t>(span) * c.raw_w * c.raw_c + 16)) <= 96 * 1024) out4[u - 1] = span;
        }
    };
    spans(cy.s0, cy.s1, d.tma_span_rows);
    {   // the period-5 row pattern of the standard 210 -> 84 resize (strided tensor copies in the TMA ingest kernel)
        bool p5 = c.obs_h % 2 == 0 && c.raw_h % 5 == 0 && 5 * (c.obs_h / 2) <= c.raw_h;
        for (int m = 0; p5 && m < c.obs_h / 2; ++m)
            p5 = cy.s0[2 * m] == 5 * m && cy.s1[2 * m] == 5 * m + 1 && cy.s0[2 * m + 1] == 5 * m + 3 && cy.s1[2 * m + 1] == 5 * m + 4;
        d.tma_period5 = p5;
        // k_ingest_gray_std: the standard ALE geometry, vertical weights (512, 1536) on even and (1536, 512) on odd rows
        bool sg = p5 && fast_ingest && c.raw_c == 1 && c.raw_h == 210 && c.raw_w == 160 && c.obs_h == 84 && c.obs_w == 84;
        for (int y = 0; sg && y < c.obs_h; ++y) {
            const int b0 = cy.coef[y] & 0xffff, b1 = cy.coef[y] >> 16;
            sg = (y & 1) ? (b0 == 1536 && b1 == 512) : (b0 == 512 && b1 == 1536);
        }
        d.std_gray = sg;
    }
    if (fast_ingest) {
        d.cx_pair = reinterpret_cast<const int4 *>(base + o_pair);
        d.cy_bs = reinterpret_cast<const int2 *>(base + o_ybs);
    }
    d.fast_squeeze = fast_squeeze;
    d.sqw_taps4 = sq_taps4;
    if (fast_squeeze) {
        d.sqw_ofs = reinterpret_cast<const int2 *>(base + o_sqofs);
        d.sqw_w = reinterpret_cast<const float *>(base + o_sqw);
        d.squeeze_q = squeeze_q;
        if (squeeze_q) d.sqw_q = base + o_sqq;
    }
    d.fast_expand = fast_expand;
    if (fast_expand) {
        d.exw_i0 = ip(o_ewi); d.exw_w0 = reinterpret_cast<const float *>(base + o_eww);
        d.exh_i0 = ip(o_ehi); d.exh_w0 = reinterpret_cast<const float *>(base + o_ehw);
        d.exw_w1 = reinterpret_cast<const float *>(base + o_eww1);
    }
    pl->dev_packed = d;
    pl->dev_packed.cy_s0 = ip(o_ys0p);
    pl->dev_packed.cy_s1 = ip(o_ys1p);
    pl->dev_packed.raw_h = static_cast<int32_t>(used.size());
    spans(ys0p, ys1p, pl->dev_packed.tma_span_rows);
    pl->dev_packed.tma_period5 = 0;   // packed rows are already gap-free
    pl->dev_packed.std_gray = 0;
    *out_plan = pl;
    return AGYM_OK;
}

int agym_plan_destroy(agym_plan *plan) {
    if (!plan) return AGYM_OK;
    if (plan->pool) cudaFree(plan->pool);
    delete plan;
    return AGYM_OK;
}

size_t agym_plan_ring_bytes(const agym_plan *plan) {
    return plan ? static_cast<size_t>(plan->cfg.n_envs) * ring_planes(plan->cfg) * plan->cfg.obs_h * plan->cfg.obs_w : 0;
}

size_t agym_plan_pcache_bytes(const agym_plan *plan) {
    return plan ? sizeof(float) * static_cast<size_t>(plan->cfg.n_envs) * ring_planes(plan->cfg) * plan->cfg.periph_h *
                      plan->cfg.periph_w
                : 0;
}

int agym_ingest_atari(const agym_plan *plan, const uint8_t *d_frames_a, const uint8_t *d_frames_b,
                      const uint8_t *d_flags, uint8_t *d_ring, int32_t *d_head, float *d_pcache, void *stream) {
    if (!plan || !d_frames_a || !d_frames_b || !d_flags || !d_ring || !d_head) return AGYM_ERR_INVALID_ARG;
    if (d_pcache && plan->cfg.periph_h == 0) return AGYM_ERR_INVALID_ARG;
    if (plan->dev.C != 1) return AGYM_ERR_UNSUPPORTED;            // ALE's grey screen is the only Atari observation
    if (plan->cfg.raw_w % 16 != 0) return AGYM_ERR_UNSUPPORTED;  // rows are staged as 16-byte vectors
    return ret(launch_ingest_atari(plan->dev, d_frames_a, d_frames_b, d_flags, d_ring, d_head, d_pcache, as_stream(stream)));
}

int agym_plan_used_rows(const agym_plan *plan, int32_t *h_rows, int32_t capacity) {
    if (!plan) return AGYM_ERR_INVALID_ARG;
    const int32_t n = static_cast<int32_t>(plan->used_rows.size());
    if (h_rows) {
        if (capacity < n) return AGYM_ERR_INVALID_ARG;
        std::memcpy(h_rows, plan->used_rows.data(), sizeof(int32_t) * n);
    }
    return n;
}

int agym_ingest_atari_packed(const agym_plan *plan, const uint8_t *d_rows_a, const uint8_t *d_rows_b,
                             const uint8_t *d_flags, uint8_t *d_ring, int32_t *d_head, float *d_pcache, void *stream) {
    if (!plan || !d_rows_a || !d_rows_b || !d_flags || !d_ring || !d_head) return AGYM_ERR_INVALID_ARG;
    if (d_pcache && plan->cfg.periph_h == 0) return AGYM_ERR_INVALID_ARG;
    if (plan->dev.C != 1) return AGYM_ERR_UNSUPPORTED;
    if (plan->cfg.raw_w % 16 != 0) return AGYM_ERR_UNSUPPORTED;
    return ret(launch_ingest_atari(plan->dev_packed, d_rows_a, d_rows_b, d_flags, d_ring, d_head, d_pcache, as_stream(stream)));
}

int agym_ingest_dmc(const agym_plan *plan, const uint8_t *d_frames, const uint8_t *d_flags, uint8_t *d_ring,
                    int32_t *d_head, float *d_pcache, void *stream) {
    if (!plan || !d_frames || !d_flags || !d_ring || !d_head) return AGYM_ERR_INVALID_ARG;
    const agym_config &c = plan->cfg;
    if (c.raw_c != 3 || c.raw_h != c.obs_h || c.raw_w != c.obs_w) return AGYM_ERR_INVALID_ARG;  // rendered at obs_size
    if (d_pcache && c.periph_h == 0) return AGYM_ERR_INVALID_ARG;
    return ret(launch_ingest_dmc(plan->dev, d_frames, d_flags, d_ring, d_head, d_pcache, as_stream(stream)));
}

int agym_stack(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, uint8_t *d_out, void *stream) {
    if (!plan || !d_ring || !d_head || !d_out) return AGYM_ERR_INVALID_ARG;
    return ret(launch_stack(plan->dev, d_ring, d_head, d_out, as_stream(stream)));
}

static int check_fov_args(const agym_plan *plan, const void *ring, const void *head, const double *action,
                          const uint8_t *ctrl, const void *loc, const void *out) {
    if (!plan || !ring || !head || !loc || !out) return AGYM_ERR_INVALID_ARG;
    if (plan->cfg.fov_h == 0) return AGYM_ERR_INVALID_ARG;
    if (!action && !ctrl) return AGYM_ERR_INVALID_ARG;  // without actions every env must be RESET / KEEP
    return AGYM_OK;
}

static int check_norm_args(const void *d_out, size_t out_bytes, const void *d_out_norm, int norm_dtype) {
    if (!d_out_norm) return AGYM_OK;
    if (norm_dtype < AGYM_DTYPE_F32 || norm_dtype > AGYM_DTYPE_BF16) return AGYM_ERR_INVALID_ARG;
    if (out_bytes % 4 != 0 || (reinterpret_cast<uintptr_t>(d_out_norm) & 15) || (reinterpret_cast<uintptr_t>(d_out) & 15))
        return AGYM_ERR_INVALID_ARG;
    return AGYM_OK;
}

int agym_observe_fixed(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, const double *d_action,
                       const uint8_t *d_fov_ctrl, int32_t *d_loc, int variant, uint8_t *d_out, void *d_out_norm,
                       int norm_dtype, void *stream) {
    int v = check_fov_args(plan, d_ring, d_head, d_action, d_fov_ctrl, d_loc, d_out);
    if (v != AGYM_OK) return v;
    if (variant < AGYM_OUT_CROP || variant > AGYM_OUT_RESIZE_FULL) return AGYM_ERR_INVALID_ARG;
    const agym_config &c = plan->cfg;
    const size_t bytes = static_cast<size_t>(c.n_envs) * ring_planes(c) * (variant == AGYM_OUT_CROP ? c.fov_h * c.fov_w : c.obs_h * c.obs_w);
    if ((v = check_norm_args(d_out, bytes, d_out_norm, norm_dtype)) != AGYM_OK) return v;
    return ret(launch_observe_fixed(plan->dev, d_ring, d_head, d_action, d_fov_ctrl, d_loc, variant, d_out, d_out_norm, norm_dtype,
                                    as_stream(stream)));
}

int agym_observe_peripheral(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, const float *d_pcache,
                            const double *d_action, const uint8_t *d_fov_ctrl, int32_t *d_loc, uint8_t *d_out,
                            void *d_out_norm, int norm_dtype, void *stream) {
    int v = check_fov_args(plan, d_ring, d_head, d_action, d_fov_ctrl, d_loc, d_out);
    if (v != AGYM_OK) return v;
    if (plan->cfg.periph_h == 0) return AGYM_ERR_INVALID_ARG;
    const agym_config &c = plan->cfg;
    if ((v = check_norm_args(d_out, static_cast<size_t>(c.n_envs) * ring_planes(c) * c.obs_h * c.obs_w, d_out_norm, norm_dtype)) != AGYM_OK) return v;
    return ret(launch_observe_peripheral(plan->dev, &plan->expand_std, d_ring, d_head, d_pcache, d_action, d_fov_ctrl, d_loc, d_out,
                                         d_out_norm, norm_dtype, as_stream(stream)));
}

int agym_observe_flexible(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, const double *d_action,
                          const int32_t *d_atype, const uint8_t *d_fov_ctrl, int32_t *d_loc, int32_t *d_res, int variant,
                          int pad_h, int pad_w, uint8_t *d_out, int32_t *d_err, void *d_out_norm, int norm_dtype, void *stream) {
    int v = check_fov_args(plan, d_ring, d_head, d_action, d_fov_ctrl, d_loc, d_out);
    if (v != AGYM_OK) return v;
    if (!d_res || variant < AGYM_OUT_CROP || variant > AGYM_OUT_RESIZE_FOV) return AGYM_ERR_INVALID_ARG;
    if (variant == AGYM_OUT_CROP && (pad_h <= 0 || pad_w <= 0 || pad_w % 4 != 0)) return AGYM_ERR_INVALID_ARG;
    const agym_config &c = plan->cfg;
    const size_t bytes = static_cast<size_t>(c.n_envs) * ring_planes(c) *
                         (variant == AGYM_OUT_CROP         ? static_cast<size_t>(pad_h) * pad_w
                          : variant == AGYM_OUT_RESIZE_FOV ? static_cast<size_t>(c.fov_h) * c.fov_w
                                                           : static_cast<size_t>(c.obs_h) * c.obs_w);
    if ((v = check_norm_args(d_out, bytes, d_out_norm, norm_dtype)) != AGYM_OK) return v;
    return ret(launch_observe_flexible(plan->dev, d_ring, d_head, nullptr, d_action, d_atype, d_fov_ctrl, d_loc, d_res, variant,
                                       pad_h, pad_w, d_out, d_err, d_out_norm, norm_dtype, as_stream(stream)));
}

int agym_observe_flexible_peripheral(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, const float *d_pcache,
                                     const double *d_action, const int32_t *d_atype, const uint8_t *d_fov_ctrl, int32_t *d_loc,
                                     int32_t *d_res, uint8_t *d_out, int32_t *d_err, void *d_out_norm, int norm_dtype, void *stream) {
    int v = check_fov_args(plan, d_ring, d_head, d_action, d_fov_ctrl, d_loc, d_out);
    if (v != AGYM_OK) return v;
    if (plan->cfg.periph_h == 0 || !d_pcache || !d_res) return AGYM_ERR_INVALID_ARG;
    const agym_config &c = plan->cfg;
    if ((v = check_norm_args(d_out, static_cast<size_t>(c.n_envs) * ring_planes(c) * c.obs_h * c.obs_w, d_out_norm, norm_dtype)) != AGYM_OK) return v;
    return ret(launch_observe_flexible(plan->dev, d_ring, d_head, d_pcache, d_action, d_atype, d_fov_ctrl, d_loc, d_res, kOutPeriph,
                                       0, 0, d_out, d_err, d_out_norm, norm_dtype, as_stream(stream)));
}

size_t agym_plan_memory_bytes(const agym_plan *plan, int depth) {
    if (!plan || plan->cfg.fov_h == 0 || depth < 1 || depth > 16) return 0;
    return static_cast<size_t>(plan->cfg.n_envs) * depth * memory_entry_bytes(plan->dev);
}

int agym_observe_fixed_memory(const agym_plan *plan, const uint8_t *d_ring, const int32_t *d_head, const double *d_action,
                              const uint8_t *d_fov_ctrl, int32_t *d_loc, int depth, uint8_t *d_mem, int32_t *d_mem_loc,
                              int32_t *d_mem_state, uint8_t *d_out, void *d_out_norm, int norm_dtype, void *stream) {
    int v = check_fov_args(plan, d_ring, d_head, d_action, d_fov_ctrl, d_loc, d_out);
    if (v != AGYM_OK) return v;
    if (depth < 1 || depth > 16 || !d_mem || !d_mem_loc || !d_mem_state) return AGYM_ERR_INVALID_ARG;
    if (reinterpret_cast<uintptr_t>(d_mem) & 15) return AGYM_ERR_INVALID_ARG;   // entries leave by bulk stores
    const agym_config &c = plan->cfg;
    if ((v = check_norm_args(d_out, static_cast<size_t>(c.n_envs) * ring_planes(c) * c.obs_h * c.obs_w, d_out_norm, norm_dtype)) != AGYM_OK) return v;
    return ret(launch_observe_fixed_memory(plan->dev, d_ring, d_head, d_action, d_fov_ctrl, d_loc, depth, d_mem, d_mem_loc,
                                           d_mem_state, d_out, d_out_norm, norm_dtype, as_stream(stream)));
}

int agym_table_cv2(int n_src, int n_dst, int zero_frac_at_border, int32_t *h_s0, int32_t *h_s1, int32_t *h_coef) {
    if (n_src <= 0 || n_dst <= 0 || !h_s0 || !h_s1 || !h_coef) return AGYM_ERR_INVALID_ARG;
    const Cv2Axis ax = build_cv2_axis(n_src, n_dst, zero_frac_at_border != 0);
    std::memcpy(h_s0, ax.s0.data(), sizeof(int32_t) * n_dst);
    std::memcpy(h_s1, ax.s1.data(), sizeof(int32_t) * n_dst);
    std::memcpy(h_coef, ax.coef.data(), sizeof(int32_t) * n_dst);
    return AGYM_OK;
}

int agym_table_aa(int n_in, int n_out, int antialias, int32_t *h_xmin, float *h_w, size_t w_capacity, int32_t *taps) {
    if (n_in <= 0 || n_out <= 0 || !h_xmin || !h_w || !taps) return AGYM_ERR_INVALID_ARG;
    const AaAxis ax = build_aa_axis(n_in, n_out, antialias != 0);
    if (ax.w.size() > w_capacity) return AGYM_ERR_INVALID_ARG;
    std::memcpy(h_xmin, ax.xmin.data(), sizeof(int32_t) * n_out);
    std::memcpy(h_w, ax.w.data(), sizeof(float) * ax.w.size());
    *taps = ax.taps;
    return AGYM_OK;
}

int agym_table_blur(int r, int f, int antialias, int32_t *h_xmin, float *h_w, uint16_t *h_q, size_t capacity, int32_t *taps,
                    int32_t *halves) {
    if (r <= 0 || f <= 0 || !h_xmin || !h_w || !h_q || !taps || !halves) return AGYM_ERR_INVALID_ARG;
    const AaAxis ax = build_blur_axis(r, f, antialias != 0);
    int nh = 1;
    const std::vector<uint32_t> q = quantize_axis_q16(ax, &nh);
    if (ax.w.size() > capacity || q.size() * 2 > capacity) return AGYM_ERR_INVALID_ARG;
    std::memcpy(h_xmin, ax.xmin.data(), sizeof(int32_t) * r);
    std::memcpy(h_w, ax.w.data(), sizeof(float) * ax.w.size());
    std::memcpy(h_q, q.data(), sizeof(uint32_t) * q.size());
    *taps = ax.taps;
    *halves = nh;
    return AGYM_OK;
}

int agym_record_step(int32_t n_envs, int is_reset, const double *d_raw_reward, const uint8_t *d_done,
                     const uint8_t *d_reset_mask, int64_t *d_ep_len, double *d_cum_reward, const int32_t *d_loc,
                     const int32_t *d_res, int32_t *d_trace_row, void *stream) {
    if (n_envs < 0 || !d_ep_len || !d_cum_reward) return AGYM_ERR_INVALID_ARG;
    return ret(launch_record_step(n_envs, is_reset, d_raw_reward, d_done, d_reset_mask, d_ep_len, d_cum_reward, d_loc, d_res,
                                  d_trace_row, as_stream(stream)));
}

int agym_normalize(const uint8_t *d_src, size_t n_bytes, int dtype, void *d_dst, void *stream) {
    if (!d_src || !d_dst || n_bytes % 16 != 0 || dtype < AGYM_DTYPE_F32 || dtype > AGYM_DTYPE_BF16) return AGYM_ERR_INVALID_ARG;
    if ((reinterpret_cast<uintptr_t>(d_src) & 15) || (reinterpret_cast<uintptr_t>(d_dst) & 15)) return AGYM_ERR_INVALID_ARG;
    return ret(launch_normalize(d_src, n_bytes, dtype, d_dst, as_stream(stream)));
}

int agym_synth_frames(uint8_t *d_dst, size_t n_bytes, uint64_t seed, void *stream) {
    if (!d_dst || n_bytes % 16 != 0) return AGYM_ERR_INVALID_ARG;
    return ret(launch_synth(d_dst, n_bytes, seed, as_stream(stream)));
}

}  // extern "C"
