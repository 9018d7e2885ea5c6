// kkt.cu — host side of the batched constrained KKT solve (row maps, dispatch, host-buffer path).
#include <algorithm>
#include <cstdio>

#include "kkt_dispatch.cuh"
#include "kkt_grad_kernels.cuh"

// ------------------------------------------------------------------ routing -------------------
// Shapes each family has an instantiation for (kkt_dispatch.cuh) and whose stage pattern it handles.
static bool tpi_has(const KktShape &s) {
    if (!s.uniform || s.d2x || s.free_final) return false;
#define X(N_, M_, A_, B_, C_) \
    if (s.n == N_ && s.m == M_ && s.P1 == A_ && (s.N == 2 || s.PM == B_) && s.PN == C_) return true;
    KKT_TPI_SIZES(X)
#undef X
    return false;
}

static bool hw_has(const KktShape &s) {
    if (!s.uniform || s.d2x || s.hess == LQRB_HESS_DENSE || s.free_final) return false;
    if (s.N < 3 || s.P1 != s.n || s.PM != 0 || s.PN != s.n) return false;
#define X(N_, M_) \
    if (s.n == N_ && s.m == M_) return true;
    KKT_HW_SIZES(X)
#undef X
    return false;
}

static bool wp_has(const KktShape &s) {
    if (s.d2x) return false;
    if (s.N < 3 || s.P1 != s.n || s.PMAX > 4 || s.PN != s.n) return false;  // up to 4 stage rows on every interior knot
#define X(N_, M_) \
    if (s.n == N_ && s.m == M_) return true;
    KKT_WP_SIZES(X)
#undef X
    return false;
}

static bool cta_has(const KktShape &s) {
    if (!s.uniform || s.d2x || s.hess == LQRB_HESS_DENSE) return false;
    if (s.N < 3 || s.P1 != s.n || s.PM > 4 || s.PN != s.n) return false;  // up to 4 stage rows on every interior knot
#define X(N_, M_) \
    if (s.n == N_ && s.m == M_) return true;
    KKT_CTA_SIZES(X)
#undef X
    return false;
}

// The tuned size class (n2, m2) a shape without a tuned kernel of its own is embedded in (see kkt_pad_maps).
static bool pad_class(const KktShape &s, int *n2, int *m2) {
    // goal rows on the whole final state, or none at all (free final state: embedded with a zero goal block)
    if (s.d2x || s.N < 3 || s.P1 != s.n || (s.PN != s.n && s.PN != 0) || s.PMAX > 4) return false;
    auto fits = [&](int N2, int M2) {
        if (N2 < s.n || M2 < s.m) return false;
        const int np = N2 - s.n, mp = M2 - s.m;
        if (np > 0 && mp < 1) return false;  // no pad control to drive the pad states
        if (np > (int64_t)(s.N - 1) * std::min(mp, np)) return false;  // every pad state must be driven at some knot
        return true;
    };
#define X(N_, M_) \
    if (fits(N_, M_)) { *n2 = N_; *m2 = M_; return true; }
    // the half-warp kernel (1.3x faster than the warp-per-instance one) exists at (8,4) and (12,4) for init + goal rows and a
    // diagonal / block-diagonal Hessian: prefer those two targets when the problem has that form
    if (s.hess != LQRB_HESS_DENSE && s.PMAX == 0 && s.PN == s.n) {
        X(8, 4) X(12, 4)
    }
    // warp-per-instance class: any Hessian mode, any stage-row count per knot
    X(8, 1) X(8, 2) X(8, 3) X(8, 4) X(12, 1) X(12, 2) X(12, 3) X(12, 4)
    if (s.hess == LQRB_HESS_DENSE || !s.uniform) return false;
    X(16, 8) X(16, 16) X(24, 8) X(24, 16) X(32, 8) X(32, 16) X(48, 16) X(64, 16)
#undef X
    return false;
}

namespace {
enum class KktFamily { Pad, Cta, Wp, Hw, Tpi, Coop };
struct KktRoute {
    KktFamily family;
    int n2 = 0, m2 = 0;  // Pad: the tuned size class
};
}  // namespace

static bool is_tuned(KktFamily f) { return f == KktFamily::Cta || f == KktFamily::Wp || f == KktFamily::Hw; }

// Which kernel family solves a shape: the only reader of the options that steer the choice.
//   kkt_variant = 2: the cooperative kernel for every shape (the tests' reference); 5: the warp-per-instance kernel
//   where the half-warp kernel also has the shape; any other value: the default.
//   kkt_pad = 0: a shape without a tuned kernel of its own goes to the cooperative kernel instead of being padded.
// The tuned kernels and the padded path read the packed data with 16-byte loads: misaligned data goes to kkt_tpi or
// kkt_coop.
static KktRoute kkt_route(const lqrb_context *h, const KktShape &s, bool data_aligned) {
    const int64_t variant = h->opt("kkt_variant", 0);
    if (variant == 2) return {KktFamily::Coop};
    if (data_aligned) {
        if (cta_has(s)) return {KktFamily::Cta};
        // for (12,4) / (8,4) block-diagonal the half-warp kernel is the faster one (49.0 vs 65.5 ms on config 5a-K)
        if (hw_has(s) && variant != 5) return {KktFamily::Hw};
        if (wp_has(s)) return {KktFamily::Wp};
    }
    if (tpi_has(s)) return {KktFamily::Tpi};
    int n2, m2;
    if (data_aligned && h->opt("kkt_pad", 1) != 0 && pad_class(s, &n2, &m2)) return {KktFamily::Pad, n2, m2};
    return {KktFamily::Coop};
}

int lqrb_kkt_tile(const lqrb_context *h, int n, int m, int N, const int32_t *p, int hess_mode,
                  int explicit_d2) {
    return kkt_route(h, make_shape(n, m, N, p, hess_mode, explicit_d2), true).family == KktFamily::Tpi ? LQRB_TILE : 1;
}

// ------------------------------------------------------------------ layout queries ------------
static int64_t knot_rows(int n, int m, int N, const int32_t *p, int hess, int d2x, int k) {
    const int mk = k < N - 1 ? m : 0, w = n + mk, p2 = k < N - 1 ? n : 0;
    return hess_rows(n, mk, hess) + w + (int64_t)p2 * w + p2 + ((d2x && k > 0) ? (int64_t)n * w : 0) +
           (int64_t)p[k] * w + p[k];
}

extern "C" int64_t lqrb_kkt_knot_offset(int32_t n, int32_t m, int32_t N, const int32_t *p,
                                        int32_t hess_mode, int32_t explicit_d2, int32_t k) {
    int64_t off = 0;
    for (int j = 0; j < k && j < N; ++j) off += knot_rows(n, m, N, p, hess_mode, explicit_d2, j);
    return off;
}

extern "C" int64_t lqrb_kkt_data_rows(int32_t n, int32_t m, int32_t N, const int32_t *p,
                                      int32_t hess_mode, int32_t explicit_d2) {
    return lqrb_kkt_knot_offset(n, m, N, p, hess_mode, explicit_d2, N);
}

// source array ids: 0 Q, 1 R, 2 Hux, 3 q, 4 r, 5 A, 6 B, 7 d, 8 D2, 9 C, 10 c
static std::vector<RowMap> kkt_data_map(const KktShape &s) {
    const int n = s.n, m = s.m, N = s.N;
    std::vector<RowMap> map;
    int Coff = 0, coff = 0, D2off = 0;
    for (int k = 0; k < N; ++k) {
        const int mk = k < N - 1 ? m : 0, w = n + mk, p2 = k < N - 1 ? n : 0, ps = s.p[k];
        // H
        if (s.hess == LQRB_HESS_DIAG) {
            for (int i = 0; i < n; ++i) map.push_back({0, k * n * n + i + i * n, 0.0});
            for (int i = 0; i < mk; ++i) map.push_back({1, k * m * m + i + i * m, 0.0});
        } else if (s.hess == LQRB_HESS_BLOCKDIAG) {
            for (int j = 0; j < n; ++j)
                for (int i = 0; i <= j; ++i) map.push_back({0, k * n * n + i + j * n, 0.0});
            for (int j = 0; j < mk; ++j)
                for (int i = 0; i <= j; ++i) map.push_back({1, k * m * m + i + j * m, 0.0});
        } else {
            for (int j = 0; j < w; ++j)
                for (int i = 0; i <= j; ++i) {
                    if (j < n)
                        map.push_back({0, k * n * n + i + j * n, 0.0});
                    else if (i < n)
                        map.push_back({2, k * m * n + (j - n) + i * m, 0.0});  // Hux'(i, j-n)
                    else
                        map.push_back({1, k * m * m + (i - n) + (j - n) * m, 0.0});
                }
        }
        // g
        for (int i = 0; i < n; ++i) map.push_back({3, k * n + i, 0.0});
        for (int i = 0; i < mk; ++i) map.push_back({4, k * m + i, 0.0});
        // D1 = [A B], d
        if (p2) {
            for (int j = 0; j < w; ++j)
                for (int i = 0; i < n; ++i) {
                    if (j < n)
                        map.push_back({5, k * n * n + i + j * n, 0.0});
                    else
                        map.push_back({6, k * n * m + i + (j - n) * n, 0.0});
                }
            for (int i = 0; i < n; ++i) map.push_back({7, k * n + i, 0.0});
        }
        if (s.d2x && k > 0) {
            for (int e = 0; e < n * w; ++e) map.push_back({8, D2off + e, 0.0});
            D2off += n * w;
        }
        for (int e = 0; e < ps * w; ++e) map.push_back({9, Coff + e, 0.0});
        for (int e = 0; e < ps; ++e) map.push_back({10, coff + e, 0.0});
        Coff += ps * w;
        coff += ps;
    }
    return map;
}

static std::vector<RowMap> identity_rows(int64_t rows) {
    std::vector<RowMap> map((size_t)rows);
    for (int64_t r = 0; r < rows; ++r) map[(size_t)r] = RowMap{0, (int32_t)r, 0.0};
    return map;
}

static std::string shape_key(const char *tag, const KktShape &s) {
    std::string k = tag;
    char buf[64];
    snprintf(buf, sizeof buf, ":%d:%d:%d:%d:%d:", s.n, s.m, s.N, s.hess, s.d2x);
    k += buf;
    for (int i = 0; i < s.N; ++i) k += std::to_string(s.p[i]) + ",";
    return k;
}

static int32_t check_kkt(lqrb_context *h, int n, int m, int N, int64_t batch, const int32_t *p, int hess) {
    if (!h) return -1;
    if (n < 1 || n > 128) return lqrb_fail(h, -2, "n out of range [1,128]");
    if (m < 1 || m > n) return lqrb_fail(h, -3, "m out of range [1,n]");
    if (N < 2) return lqrb_fail(h, -4, "N must be >= 2");
    if (batch < 0) return lqrb_fail(h, -5, "batch must be >= 0");
    if (!p) return lqrb_fail(h, -6, "p is NULL");
    for (int k = 0; k < N; ++k)
        if (p[k] < 0 || p[k] > n + m) return lqrb_fail(h, -6, "p[k] out of range [0, n+m]");
    if (hess < 0 || hess > 2) return lqrb_fail(h, -7, "hess_mode must be 0, 1 or 2");
    return 0;
}

// ------------------------------------------------------------------ tuned families ------------
// The conditioning record of one API call (lqrb_kkt_last_condition), over every chunk its tuned kernels ran in:
// scratch chunks, padded chunks and host-buffer chunks append in instance order.
namespace {
struct KktRecord {
    std::vector<int32_t> cond;  // log2 pivot ratio per instance
    int64_t refined = 0;        // instances re-solved by the Cholesky-based kernel
    bool tuned = false;         // a tuned kernel ran
};
}  // namespace

// A call that ran no tuned kernel leaves the handle's record as it was; with kkt_refine = 0 only the count is reset.
static void kkt_keep_record(lqrb_context *h, KktRecord &rec) {
    if (!rec.tuned) return;
    h->last_refined = rec.refined;
    if (!rec.cond.empty()) h->last_cond.swap(rec.cond);
}

// The tuned large-size kernels (kkt_hw2, kkt_wp, kkt_cta) carry the block elimination with explicit SPD inverses
// (products instead of the reference's sequential triangular solves); their error grows with cond(Sigma_k) where the
// reference's U'U form (src/cholesky_solve.jl:47-67) does not.  The kernels report, per instance, log2 of the worst
// pivot ratio met in any Sigma_k (free: integer compares of the pivots' high words).  Instances above `kkt_cond_bits`
// are solved again by the Cholesky-based general kernel — the reference's own operation order — which overwrites their
// outputs.  `kkt_refine` = 0 switches this off.  Costs one 4-byte-per-instance read-back and a stream synchronisation.
static int32_t kkt_resolve_ill_conditioned(lqrb_context *h, const KktShape &s, int64_t cb, int flags, const double *dc,
                                           const int32_t *cinfo_dev, double *dz, double *mult, double *res, int32_t *info,
                                           Lane lane, KktRecord *record) {
    if (h->opt("kkt_refine", 1) == 0) return 0;
    const cudaStream_t st = lane.stream;
    int32_t *hc = (int32_t *)lqrb_pinned(h, lane.index, (size_t)cb * sizeof(int32_t));
    if (!hc) return 1000 + (int)cudaErrorMemoryAllocation;
    LQRB_CUDA(h, cudaMemcpyAsync(hc, cinfo_dev, (size_t)cb * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    LQRB_CUDA(h, cudaStreamSynchronize(st));
    record->cond.insert(record->cond.end(), hc, hc + cb);
    const int thr = (int)h->opt("kkt_cond_bits", LQRB_KKT_COND_BITS);
    std::vector<int32_t> list;
    for (int64_t i = 0; i < cb; ++i)
        if (hc[i] >= thr) list.push_back((int32_t)i);
    if (list.empty()) return 0;
    const KktSizes z = kkt_sizes(s);
    // the general kernel keeps full-storage records: process the list in pieces that fit the scratch budget
    const size_t per = (size_t)z.rec_rows * 8;
    const int64_t piece = std::max<int64_t>(1, (int64_t)(((size_t)h->opt("scratch_budget_mb", 49152) << 20) / 4 / per));
    for (size_t first = 0; first < list.size(); first += (size_t)piece) {
        const int64_t cnt = std::min<int64_t>(piece, (int64_t)(list.size() - first));
        int32_t *dl = (int32_t *)lqrb_scratch(h, SCR_REFINE_LIST, (size_t)cb * sizeof(int32_t), lane.index);
        double *rec = (double *)lqrb_scratch(h, SCR_REFINE, (size_t)std::min<int64_t>(piece, cb) * per, lane.index);
        if (!dl || !rec) return 1000 + (int)cudaErrorMemoryAllocation;
        LQRB_CUDA(h, cudaMemcpyAsync(dl, list.data() + first, (size_t)cnt * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        KktCoopExtra ex;
        ex.list = dl;
        std::vector<int32_t> pf;
        const int32_t *pp = s.p;
        if (s.free_final) {  // the general kernel solves the problem as it is (no goal rows) inside the tuned kernel's layout
            pf.assign(s.p, s.p + s.N);
            pf[s.N - 1] = 0;
            pp = pf.data();
            ex.data_stride = z.data_rows;
            ex.mult_stride = z.P;
        }
        int32_t rc = launch_kkt_coop(h, s.n, s.m, s.N, pp, s.hess, s.d2x, flags, cnt, dc, rec, dz, mult, res, info, lane, &ex);
        if (rc) return rc;
        LQRB_CUDA(h, cudaStreamSynchronize(st));  // `list` (pageable) must outlive the copy
    }
    record->refined += (int64_t)list.size();
    return 0;
}

// scratch of the tuned kernels in doubles: the largest need of the families that have this (n, m)
static size_t kkt_tuned_scratch_doubles(const KktShape &s, int64_t batch) {
    const size_t per = std::max(kkt_cta_scratch_per_instance(s), std::max(kkt_hw_scratch_per_instance(s), kkt_wp_scratch_per_instance(s)));
    return per == 0 ? 0 : (size_t)batch * per + 2;
}

// The tuned large-size kernels keep records and pre-pass results in scratch (2.5 MB per instance for n=12,
// N=1001; 13.7 MB for n=64, N=101).  Batches are processed in chunks so that the scratch stays under
// `scratch_budget_mb` (default 48 GB of the 180 GB) whatever the batch size.  A chunk is a whole number of
// resident waves of the sequential kernel (its CTAs live for the whole horizon, so a partial wave is a tail).
static int64_t kkt_tuned_chunk(const lqrb_context *h, const KktShape &s) {
    const size_t per = kkt_tuned_scratch_doubles(s, 1);
    if (per == 0) return 0;
    const size_t budget = (size_t)h->opt("scratch_budget_mb", 49152) << 20;
    int64_t c = (int64_t)(budget / (per * 8));
    // kkt_hw: 3 CTAs x 8 instances per SM; kkt_cta: 2 CTAs x 1 instance per SM
    const int64_t wave = (int64_t)h->sm_count * (s.n + s.m <= 16 ? 24 : 2);
    c = std::max<int64_t>(wave, c / wave * wave);
    return c;
}

// scratch of a tuned family for `batch` instances (never less than the general kernel needs)
static size_t kkt_tuned_scratch_bytes(const lqrb_context *h, const KktShape &s, const KktSizes &z, int64_t batch) {
    return std::max((size_t)lqrb_padded_batch(batch) * z.rec_rows * 8,
                    kkt_tuned_scratch_doubles(s, std::min(batch, kkt_tuned_chunk(h, s))) * 8 + 64);
}

// Runs a tuned family over the batch in chunks of kkt_tuned_chunk instances, each followed by the re-solve of its
// ill-conditioned instances.  The kernel name counts the re-solved instances of the whole call so far.
static int32_t kkt_solve_tuned(lqrb_context *h, KktFamily family, const KktShape &s, int64_t batch, int flags,
                               const double *data, double *scratch, double *dz, double *mult, double *res, int32_t *info,
                               Lane lane, KktRecord *record) {
    auto launch = family == KktFamily::Cta ? kkt_cta_chunk : family == KktFamily::Wp ? kkt_wp_chunk : kkt_hw_chunk;
    const KktSizes z = kkt_sizes(s);
    const int soc = (flags & LQRB_FLAG_SOC) ? 1 : 0;
    const int64_t chunk = std::min(batch, kkt_tuned_chunk(h, s));
    std::string name;
    for (int64_t first = 0; first < batch; first += chunk) {
        const int64_t cb = std::min(chunk, batch - first);
        const double *dc = data + first * z.data_rows;
        double *dzc = dz + first * z.NN, *mc = mult + first * z.P, *rc_ = res ? res + first * z.NN : nullptr;
        int32_t *ic = info ? info + first : nullptr, *cinfo = nullptr;
        int32_t rc = launch(h, s, cb, soc, dc, scratch, dzc, mc, rc_, ic, &cinfo, lane.stream);
        if (rc) return rc;
        name = h->kernel_name;  // (the re-solve names its own kernel)
        rc = kkt_resolve_ill_conditioned(h, s, cb, soc ? LQRB_FLAG_SOC : 0, dc, cinfo, dzc, mc, rc_, ic, lane, record);
        if (rc) return rc;
    }
    record->tuned = true;
    h->kernel_name = name;
    if (record->refined) h->kernel_name += "+kkt_coop[" + std::to_string(record->refined) + " ill-conditioned]";
    return 0;
}

// ------------------------------------------------------------------ padding into a tuned size class ----
// A shape without a tuned kernel of its own (n = 7, 9..11, 13.., m > 4, ...) is embedded in the next tuned size class
// (n2, m2) instead of falling to the general kernel (14-50x slower): pad states xp with cost I, dynamics
// xp_{k+1} = xp_k + (pad control c drives pad state (k mp + c) mod np at knot k: every pad state is driven at some knot,
// so the pad part of the goal rows stays independent of the dynamics rows), init / goal rows xp_1 = xp_N = 0, pad
// controls with cost I.  The pad
// variables and their multipliers are exactly zero at the optimum and the original variables see the same KKT system.
// The packed data (layout of s) is expanded on the device into the layout of the padded shape, the tuned kernel runs,
// and dz, mult, res are compacted back: two extra passes over the data, a few percent of what the padding saves.
namespace {
struct PadMaps {
    std::vector<RowMap> data, dz, mult;  // rows of the padded layout -> offset in the original one (or fill / skip)
};
}

static PadMaps kkt_pad_maps(const KktShape &s, int n2, int m2) {
    const int n = s.n, m = s.m, N = s.N, np = n2 - n, mpe = std::min(m2 - m, np);  // pad controls in use
    PadMaps M;
    int64_t base = 0;  // start of knot k in the original packed record
    int64_t moff = 0;  // original multiplier offset
    for (int k = 0; k < N; ++k) {
        const bool first = k == 0, last = k == N - 1;
        const int mk = last ? 0 : m, w = n + mk, p2 = last ? 0 : n, ps = s.p[k];
        const int mk2 = last ? 0 : m2, w2 = n2 + mk2;
        const int64_t oH = base, og = oH + hess_rows(n, mk, s.hess), oD1 = og + w, od = oD1 + (int64_t)p2 * w, oC = od + p2,
                      oc = oC + (int64_t)ps * w;
        // padded z index -> original z index (-1: pad)
        auto zmap = [&](int j) { return j < n ? j : (j < n2 ? -1 : (j - n2 < mk ? n + (j - n2) : -1)); };
        auto src = [&](int64_t off) { M.data.push_back(RowMap{0, (int32_t)off, 0.0}); };
        auto fill = [&](double v) { M.data.push_back(RowMap{-1, 0, v}); };
        // H
        if (s.hess == LQRB_HESS_DIAG) {
            for (int j = 0; j < w2; ++j) {
                const int o = zmap(j);
                if (o >= 0) src(oH + o); else fill(1.0);
            }
        } else if (s.hess == LQRB_HESS_BLOCKDIAG) {
            for (int j = 0; j < n2; ++j)
                for (int i = 0; i <= j; ++i) {
                    if (j < n) src(oH + (int64_t)j * (j + 1) / 2 + i); else fill(i == j ? 1.0 : 0.0);
                }
            for (int j = 0; j < mk2; ++j)
                for (int i = 0; i <= j; ++i) {
                    if (j < mk) src(oH + tri(n) + (int64_t)j * (j + 1) / 2 + i); else fill(i == j ? 1.0 : 0.0);
                }
        } else {
            for (int j = 0; j < w2; ++j)
                for (int i = 0; i <= j; ++i) {
                    const int oi = zmap(i), oj = zmap(j);
                    if (oi >= 0 && oj >= 0) src(oH + (int64_t)oj * (oj + 1) / 2 + oi); else fill(i == j ? 1.0 : 0.0);
                }
        }
        // g
        for (int j = 0; j < w2; ++j) {
            const int o = zmap(j);
            if (o >= 0) src(og + o); else fill(0.0);
        }
        // D1 = [A B] (n2 x w2 column-major), d
        if (!last) {
            for (int j = 0; j < w2; ++j)
                for (int i = 0; i < n2; ++i) {
                    const int o = zmap(j);
                    if (i < n) {
                        if (o >= 0) src(oD1 + i + (int64_t)o * n); else fill(0.0);
                    } else {
                        const int r = i - n, c = j - n2 - m;  // pad state r, pad control c (if 0 <= c < mpe)
                        fill((j == i || (c >= 0 && c < mpe && (k * mpe + c) % np == r)) ? 1.0 : 0.0);
                    }
                }
            for (int i = 0; i < n2; ++i) {
                if (i < n) src(od + i); else fill(0.0);
            }
        }
        // C, c : the end knots have n rows (+ identity rows on the pad states), the interior ones their ps rows
        const int ps2 = (first || last) ? n2 : ps;
        const bool nogoal = last && ps == 0;  // free final state: a zero goal block (the kernel leaves mu_N = 0)
        for (int j = 0; j < w2; ++j)
            for (int i = 0; i < ps2; ++i) {
                const int o = zmap(j);
                if (i < ps) {
                    if (o >= 0) src(oC + i + (int64_t)o * ps); else fill(0.0);
                } else {
                    fill((!nogoal && j == n + (i - ps)) ? 1.0 : 0.0);  // (first / last knot: ps = n) pad state i - n pinned to 0
                }
            }
        for (int i = 0; i < ps2; ++i) {
            if (i < ps) src(oc + i); else fill(0.0);
        }
        base = oc + ps;
        // outputs: dz / res rows of knot k
        for (int j = 0; j < w2; ++j) {
            const int o = zmap(j);
            M.dz.push_back(o >= 0 ? RowMap{0, (int32_t)((int64_t)k * (n + m) + o), 0.0} : RowMap{-1, 0, 0.0});
        }
        // multipliers: [mu_k (ps2); lam_k (n2)]
        for (int i = 0; i < ps2; ++i) M.mult.push_back(i < ps ? RowMap{0, (int32_t)(moff + i), 0.0} : RowMap{-1, 0, 0.0});
        moff += ps;
        if (!last) {
            for (int i = 0; i < n2; ++i) M.mult.push_back(i < n ? RowMap{0, (int32_t)(moff + i), 0.0} : RowMap{-1, 0, 0.0});
            moff += n;
        }
    }
    return M;
}

struct PadPlan {
    std::vector<int32_t> p2;
    KktShape s2;
    KktSizes z2;
    int64_t chunk;
    size_t data_b, out_b, scr_b;  // bytes per chunk: padded data | dz2, mult2, res2 | scratch of the tuned kernel
};

static void kkt_pad_plan(const lqrb_context *h, const KktShape &s, int n2, int m2, int64_t batch, PadPlan *P) {
    P->p2.assign(s.p, s.p + s.N);
    P->p2[0] = n2;
    P->p2[s.N - 1] = n2;
    P->s2 = make_shape(n2, m2, s.N, P->p2.data(), s.hess, 0);
    P->s2.free_final = s.PN == 0;
    P->z2 = kkt_sizes(P->s2);
    P->chunk = std::max<int64_t>(1, std::min(batch, kkt_tuned_chunk(h, P->s2)));
    const size_t ldb = (size_t)lqrb_padded_batch(P->chunk);
    P->data_b = (ldb * P->z2.data_rows * 8 + 255) / 256 * 256;
    P->out_b = (ldb * (2 * P->z2.NN + P->z2.P) * 8 + 255) / 256 * 256;
    P->scr_b = (kkt_tuned_scratch_bytes(h, P->s2, P->z2, P->chunk) + 255) / 256 * 256;
}

// info codes of the padded shape -> the caller's z numbering.  The pad states sit between the caller's states and its
// controls (zmap above), so a Hessian pivot (stage 0) above n2 is a control and moves down by n2 - n; the Schur blocks
// list the caller's rows first and keep their numbers.
__global__ void kkt_unpad_info_kernel(int32_t *info, int64_t cb, int n, int n2) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cb) return;
    const int32_t c = info[i], pivot = c % 1000;
    if (c > 0 && pivot < 100 && pivot > n2) info[i] = c - (n2 - n);
}

static int32_t kkt_solve_padded(lqrb_context *h, const KktShape &s, int n2, int m2, int64_t batch, int flags,
                                const double *data, double *scratch, double *dz, double *mult, double *res, int32_t *info,
                                Lane lane, KktRecord *record) {
    const cudaStream_t st = lane.stream;
    PadPlan P;
    kkt_pad_plan(h, s, n2, m2, batch, &P);
    const KktFamily family = kkt_route(h, P.s2, true).family;
    if (!is_tuned(family)) return lqrb_fail(h, 1, "padded KKT shape has no tuned kernel");
    const KktSizes z = kkt_sizes(s);
    char key[64];
    snprintf(key, sizeof key, "->%d,%d", n2, m2);
    const std::string k0 = shape_key("pad", s) + key;
    DevMap md, mz, mm;
    if (h->maps.find(k0 + ":m") == h->maps.end()) {  // first use of this shape: build and upload the three maps
        const PadMaps M = kkt_pad_maps(s, n2, m2);
        md = lqrb_get_map(h, k0 + ":d", M.data);
        mz = lqrb_get_map(h, k0 + ":z", M.dz);
        mm = lqrb_get_map(h, k0 + ":m", M.mult);
    } else {
        md = h->maps[k0 + ":d"];
        mz = h->maps[k0 + ":z"];
        mm = h->maps[k0 + ":m"];
    }
    if (md.rows != P.z2.data_rows || mz.rows != P.z2.NN || mm.rows != P.z2.P) return lqrb_fail(h, 1, "pad map size mismatch");
    char *base = reinterpret_cast<char *>(scratch);
    double *data2 = reinterpret_cast<double *>(base);
    double *dz2 = reinterpret_cast<double *>(base + P.data_b);
    const size_t ldb = (size_t)lqrb_padded_batch(P.chunk);
    double *mult2 = dz2 + ldb * P.z2.NN, *res2 = mult2 + ldb * P.z2.P;
    double *scr2 = reinterpret_cast<double *>(base + P.data_b + P.out_b);
    for (int64_t first = 0; first < batch; first += P.chunk) {
        const int64_t cb = std::min(P.chunk, batch - first);
        ArrayTable src = {};
        src.ptr[0] = data + first * z.data_rows;
        src.stride[0] = z.data_rows;
        int32_t rc = lqrb_gather_pack(h, md, src, cb, 1, data2, st);
        if (rc) return rc;
        rc = kkt_solve_tuned(h, family, P.s2, cb, flags, data2, scr2, dz2, mult2, res ? res2 : nullptr,
                             info ? info + first : nullptr, lane, record);
        if (rc) return rc;
        if (info) {
            kkt_unpad_info_kernel<<<(unsigned)((cb + 255) / 256), 256, 0, st>>>(info + first, cb, s.n, n2);
            LQRB_CUDA(h, cudaGetLastError());
        }
        ArrayTableOut o = {};
        o.ptr[0] = dz + first * z.NN;
        o.stride[0] = z.NN;
        rc = lqrb_scatter_unpack(h, mz, o, cb, 1, dz2, st);
        if (rc) return rc;
        if (res) {
            o.ptr[0] = res + first * z.NN;
            rc = lqrb_scatter_unpack(h, mz, o, cb, 1, res2, st);
            if (rc) return rc;
        }
        o.ptr[0] = mult + first * z.P;
        o.stride[0] = z.P;
        rc = lqrb_scatter_unpack(h, mm, o, cb, 1, mult2, st);
        if (rc) return rc;
    }
    char nm[64];
    snprintf(nm, sizeof nm, " <- (%d,%d)%s padded", s.n, s.m, s.PN == 0 ? " free final state" : "");
    h->kernel_name += nm;
    return 0;
}

// scratch of one call, sized for 16-byte aligned data (misaligned data runs the general kernel, which needs less)
static size_t kkt_scratch_bytes(const lqrb_context *h, const KktShape &s, const KktSizes &z, int64_t batch) {
    const KktRoute r = kkt_route(h, s, true);
    const size_t general = (size_t)lqrb_padded_batch(batch) * z.rec_rows * 8;
    if (r.family == KktFamily::Pad) {
        PadPlan P;
        kkt_pad_plan(h, s, r.n2, r.m2, batch, &P);
        return std::max(P.data_b + P.out_b + P.scr_b, general);
    }
    return is_tuned(r.family) ? kkt_tuned_scratch_bytes(h, s, z, batch) : general;
}

static int32_t kkt_solve_on(lqrb_context *h, const KktShape &s, int64_t batch, int flags,
                            const double *data, double *scratch, double *dz, double *mult, double *res,
                            int32_t *info, Lane lane, KktRecord *record) {
    if (batch == 0) return 0;
    const KktRoute r = kkt_route(h, s, ((uintptr_t)data & 15) == 0);
    switch (r.family) {
    case KktFamily::Pad:
        return kkt_solve_padded(h, s, r.n2, r.m2, batch, flags, data, scratch, dz, mult, res, info, lane, record);
    case KktFamily::Cta:
    case KktFamily::Wp:
    case KktFamily::Hw:
        return kkt_solve_tuned(h, r.family, s, batch, flags, data, scratch, dz, mult, res, info, lane, record);
    case KktFamily::Tpi:
        return kkt_launch_tpi(h, s, batch, flags, data, scratch, dz, mult, res, info, lane.stream);
    case KktFamily::Coop:
        break;
    }
    return launch_kkt_coop(h, s.n, s.m, s.N, s.p, s.hess, s.d2x, flags, batch, data, scratch, dz, mult, res,
                           info, lane);
}

int32_t lqrb_kkt_solve_packed_on(lqrb_context *h, int n, int m, int N, int64_t batch, const int32_t *p, int hess_mode,
                                 int explicit_d2, int flags, const double *data, double *dz, double *mult, double *res,
                                 int32_t *info, Lane lane) {
    const KktShape s = make_shape(n, m, N, p, hess_mode, explicit_d2);
    const KktSizes z = kkt_sizes(s);
    double *scratch = (double *)lqrb_scratch(h, SCR_FACT, kkt_scratch_bytes(h, s, z, batch), lane.index);
    if (!scratch) return 1000 + (int)cudaErrorMemoryAllocation;
    KktRecord record;
    int32_t rc = kkt_solve_on(h, s, batch, flags, data, scratch, dz, mult, res, info, lane, &record);
    if (rc) return rc;
    kkt_keep_record(h, record);
    return 0;
}

extern "C" int32_t lqrb_kkt_solve_packed_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N,
                                             int64_t batch, const int32_t *p, int32_t hess_mode,
                                             int32_t explicit_d2, int32_t flags, const double *data,
                                             double *dz, double *mult, double *res, int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!data) return lqrb_fail(h, -11, "data is NULL");
    if (!dz) return lqrb_fail(h, -12, "dz is NULL");
    if (!mult) return lqrb_fail(h, -13, "mult is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    return lqrb_kkt_solve_packed_on(h, n, m, N, batch, p, hess_mode, explicit_d2, flags, data, dz, mult, res, info,
                                    Lane{h->stream, 0});
}

// ------------------------------------------------------------------ pack / unpack -------------
static int32_t kkt_pack_on(lqrb_context *h, const KktShape &s, const KktSizes &z, int64_t batch,
                           const double *const src[11], double *data, cudaStream_t st) {
    const int n = s.n, m = s.m, N = s.N;
    const int64_t strides[11] = {(int64_t)n * n * N, (int64_t)m * m * (N - 1), (int64_t)m * n * (N - 1),
                                 (int64_t)n * N,     (int64_t)m * (N - 1),     (int64_t)n * n * (N - 1),
                                 (int64_t)n * m * (N - 1), (int64_t)n * (N - 1), z.sD2, z.sC, z.sc};
    ArrayTable t = {};
    for (int i = 0; i < 11; ++i) {
        t.ptr[i] = src[i];
        t.stride[i] = strides[i];
    }
    const int tile = lqrb_kkt_tile(h, n, m, N, s.p, s.hess, s.d2x);
    return lqrb_gather_pack(h, lqrb_get_map(h, shape_key("kd", s), kkt_data_map(s)), t, batch, tile, data, st);
}

extern "C" int32_t lqrb_kkt_pack_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                     const int32_t *p, int32_t hess_mode, const double *Q,
                                     const double *R, const double *Hux, const double *q,
                                     const double *r, const double *A, const double *B,
                                     const double *d, const double *D2, const double *C,
                                     const double *c, double *data) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!Q || !R || !q || !r || !A || !B || !d) return lqrb_fail(h, -8, "a required input array is NULL");
    if (!data) return lqrb_fail(h, -19, "data is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, D2 != nullptr);
    const KktSizes z = kkt_sizes(s);
    if (z.sC > 0 && (!C || !c)) return lqrb_fail(h, -17, "C/c is NULL but p has non-zero entries");
    const double *src[11] = {Q, R, Hux, q, r, A, B, d, D2, C, c};
    return kkt_pack_on(h, s, z, batch, src, data, h->stream);
}

static int32_t kkt_unpack_on(lqrb_context *h, const KktShape &s, const KktSizes &z, int64_t batch,
                             const double *dzp, const double *multp, const double *resp, double *dz,
                             double *mult, double *res, cudaStream_t st) {
    const int tile = lqrb_kkt_tile(h, s.n, s.m, s.N, s.p, s.hess, s.d2x);
    ArrayTableOut t = {};
    t.ptr[0] = dz;
    t.stride[0] = z.NN;
    int32_t rc = lqrb_scatter_unpack(h, lqrb_get_map(h, "id" + std::to_string(z.NN), identity_rows(z.NN)), t,
                                     batch, tile, dzp, st);
    if (rc) return rc;
    t.ptr[0] = mult;
    t.stride[0] = z.P;
    rc = lqrb_scatter_unpack(h, lqrb_get_map(h, "id" + std::to_string(z.P), identity_rows(z.P)), t, batch,
                             tile, multp, st);
    if (rc || !res) return rc;
    t.ptr[0] = res;
    t.stride[0] = z.NN;
    return lqrb_scatter_unpack(h, lqrb_get_map(h, "id" + std::to_string(z.NN), identity_rows(z.NN)), t, batch,
                               tile, resp, st);
}

extern "C" int32_t lqrb_kkt_tile_width(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, const int32_t *p,
                                       int32_t hess_mode, int32_t explicit_d2) {
    int32_t rc = check_kkt(h, n, m, N, 0, p, hess_mode);
    if (rc) return rc;
    return lqrb_kkt_tile(h, n, m, N, p, hess_mode, explicit_d2);
}

extern "C" int32_t lqrb_kkt_unpack_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                       const int32_t *p, int32_t hess_mode, int32_t explicit_d2,
                                       const double *dzp, const double *multp, const double *resp, double *dz,
                                       double *mult, double *res) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!dzp || !multp) return lqrb_fail(h, -9, "packed dz / mult is NULL");
    if (!dz || !mult) return lqrb_fail(h, -12, "dz / mult is NULL");
    if (res && !resp) return lqrb_fail(h, -11, "res requested but the packed res is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, explicit_d2);
    const KktSizes z = kkt_sizes(s);
    return kkt_unpack_on(h, s, z, batch, dzp, multp, resp, dz, mult, res, h->stream);
}

// ------------------------------------------------------------------ full call -----------------
// The instance-major inputs of a KKT call (sources of kkt_data_map, NULL where absent) with their bytes per instance;
// an absent Hux or D2 counts as 0 bytes.
static std::vector<HostArray> kkt_inputs(const KktShape &s, const KktSizes &z, const double *const src[11]) {
    const int64_t n = s.n, m = s.m, N = s.N, K1 = N - 1;
    const int64_t per[11] = {n * n * N, m * m * K1, src[2] ? m * n * K1 : 0, n * N,  m * K1, n * n * K1,
                             n * m * K1, n * K1,     src[8] ? z.sD2 : 0,     z.sC,   z.sc};
    std::vector<HostArray> v(11);
    for (int i = 0; i < 11; ++i) v[i] = {src[i], per[i] * 8};
    return v;
}

// gather sources of one chunk: the driver's device pointers with the listed arrays' strides
static ArrayTable kkt_array_table(const std::vector<HostArray> &inputs, const void *const *in) {
    ArrayTable t = {};
    for (size_t i = 0; i < inputs.size(); ++i) {
        t.ptr[i] = (const double *)in[i];
        t.stride[i] = inputs[i].bytes / 8;
    }
    return t;
}

extern "C" int32_t lqrb_kkt_solve_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                      const int32_t *p, int32_t hess_mode, int32_t flags,
                                      const double *Q, const double *R, const double *Hux,
                                      const double *q, const double *r, const double *A,
                                      const double *B, const double *d, const double *D2,
                                      const double *C, const double *c, double *dz, double *mult,
                                      double *res, int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!Q || !R || !q || !r || !A || !B || !d) return lqrb_fail(h, -9, "a required input array is NULL");
    if (!dz) return lqrb_fail(h, -20, "dz is NULL");
    if (!mult) return lqrb_fail(h, -21, "mult is NULL");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, D2 != nullptr);
    const KktSizes z = kkt_sizes(s);
    if (z.sC > 0 && (!C || !c)) return lqrb_fail(h, -18, "C/c is NULL but p has non-zero entries");
    const double *src[11] = {Q, R, Hux, q, r, A, B, d, D2, C, c};
    KktRecord record;
    rc = lqrb_for_chunks(
        h, batch, 0, kkt_inputs(s, z, src), {{dz, z.NN * 8}, {mult, z.P * 8}, {res, z.NN * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const int64_t ldb = lqrb_padded_batch(cb);
            double *data = (double *)lqrb_scratch(h, SCR_PACK_IN, (size_t)ldb * z.data_rows * 8, lane.index);
            double *dzp = (double *)lqrb_scratch(h, SCR_PACK_OUT, (size_t)ldb * z.NN * 8, lane.index);
            double *mp = (double *)lqrb_scratch(h, SCR_PACK_OUT2, (size_t)ldb * z.P * 8, lane.index);
            double *rp = out[2] ? (double *)lqrb_scratch(h, SCR_PACK_OUT3, (size_t)ldb * z.NN * 8, lane.index) : nullptr;
            double *scr = (double *)lqrb_scratch(h, SCR_FACT, kkt_scratch_bytes(h, s, z, cb), lane.index);
            if (!data || !dzp || !mp || !scr || (out[2] && !rp)) return 1000 + (int)cudaErrorMemoryAllocation;
            int32_t rc = kkt_pack_on(h, s, z, cb, (const double *const *)in, data, lane.stream);
            if (rc) return rc;
            rc = kkt_solve_on(h, s, cb, flags, data, scr, dzp, mp, rp, (int32_t *)out[3], lane, &record);
            if (rc) return rc;
            return kkt_unpack_on(h, s, z, cb, dzp, mp, rp, (double *)out[0], (double *)out[1], (double *)out[2],
                                 lane.stream);
        });
    if (rc) return rc;
    kkt_keep_record(h, record);
    return 0;
}

// ------------------------------------------------------------------ gradient ------------------
// The adjoint problem of lqrb_kkt_grad_f64 (DESIGN §4.9): the forward matrices, with g taken from dz_bar (Primals
// order) and d, c from mult_bar (order [mu_1; lam_1; ...; mu_N]).  Source ids as kkt_data_map with 3 = dz_bar and
// 7 = mult_bar (4 and 10 unused); a NULL source packs zeros.
static std::vector<RowMap> kkt_adjoint_data_map(const KktShape &s) {
    const int n = s.n, m = s.m;
    std::vector<int32_t> lam((size_t)s.N), mu_of_c;  // multiplier offset of lam_k | of each row of the concatenated c
    int32_t off = 0;
    for (int k = 0; k < s.N; ++k) {
        for (int e = 0; e < s.p[k]; ++e) mu_of_c.push_back(off + e);
        off += s.p[k];
        lam[(size_t)k] = off;
        if (k < s.N - 1) off += n;
    }
    std::vector<RowMap> map = kkt_data_map(s);
    for (RowMap &r : map) {
        const int32_t o = r.offset;
        if (r.array == 3) r = RowMap{3, o / n * (n + m) + o % n, 0.0};  // q_k(i) -> x_k(i)
        else if (r.array == 4) r = RowMap{3, o / m * (n + m) + n + o % m, 0.0};  // r_k(i) -> u_k(i)
        else if (r.array == 7) r = RowMap{7, lam[(size_t)(o / n)] + o % n, 0.0};
        else if (r.array == 10) r = RowMap{7, mu_of_c[(size_t)o], 0.0};
    }
    return map;
}

// per-knot offset tables of the gradient kernel (KktGradTables), built once per shape
static int32_t kkt_grad_tables(lqrb_context *h, const KktShape &s, KktGradTables *t) {
    const int n = s.n, m = s.m, N = s.N;
    const std::string key = shape_key("kgrad", s);
    auto it = h->blobs.find(key);
    int32_t *d = nullptr;
    if (it != h->blobs.end()) {
        d = (int32_t *)it->second;
    } else {
        std::vector<int32_t> host(5 * (size_t)(N + 1), 0);
        int32_t *mu = host.data(), *lam = mu + N + 1, *C = lam + N + 1, *c = C + N + 1, *D2 = c + N + 1;
        for (int k = 0; k < N; ++k) {
            const int w = n + (k < N - 1 ? m : 0);
            lam[k] = mu[k] + s.p[k];
            mu[k + 1] = lam[k] + (k < N - 1 ? n : 0);
            C[k + 1] = C[k] + s.p[k] * w;
            c[k + 1] = c[k] + s.p[k];
            if (k > 0) D2[k + 1] = D2[k] + n * w;
        }
        lam[N] = mu[N];
        LQRB_CUDA(h, cudaMalloc(&d, host.size() * sizeof(int32_t)));
        LQRB_CUDA(h, cudaMemcpy(d, host.data(), host.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        LQRB_CUDA(h, cudaStreamSynchronize(cudaStreamLegacy));  // pageable source: wait for the staged DMA
        h->blobs[key] = d;
    }
    *t = KktGradTables{d, d + (N + 1), d + 2 * (N + 1), d + 3 * (N + 1), d + 4 * (N + 1)};
    return 0;
}

// Gradient of l(dz, mult) through lqrb_kkt_solve_f64 (DESIGN §4.9): the adjoint problem (same matrices, right-hand
// side from the cotangents) is packed and solved by the forward dispatch, its solution unpacked to instance-major
// scratch, and kkt_grad_kernel forms every requested gradient from the two solutions.  The adjoint solve's
// conditioning record is dropped: lqrb_kkt_last_condition keeps describing the last forward solve.
extern "C" int32_t lqrb_kkt_grad_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                     const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                                     const double *R, const double *Hux, const double *A, const double *B,
                                     const double *D2, const double *C, const double *dz, const double *mult,
                                     const double *dz_bar, const double *mult_bar, double *gQ, double *gR,
                                     double *gHux, double *gq, double *gr, double *gA, double *gB, double *gd,
                                     double *gD2, double *gC, double *gc, int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (flags & LQRB_FLAG_SOC) return lqrb_fail(h, -8, "flags: the gradient of the second-order correction is not provided");
    if (flags) return lqrb_fail(h, -8, "flags must be 0");
    if (!Q) return lqrb_fail(h, -9, "Q is NULL");
    if (!R) return lqrb_fail(h, -10, "R is NULL");
    if (!A) return lqrb_fail(h, -12, "A is NULL");
    if (!B) return lqrb_fail(h, -13, "B is NULL");
    const KktShape s = make_shape(n, m, N, p, hess_mode, D2 != nullptr);
    const KktSizes z = kkt_sizes(s);
    if (z.sC > 0 && !C) return lqrb_fail(h, -15, "C is NULL but p has non-zero entries");
    if (!dz) return lqrb_fail(h, -16, "dz is NULL");
    if (!mult) return lqrb_fail(h, -17, "mult is NULL");
    if (!dz_bar && !mult_bar) return lqrb_fail(h, -18, "dz_bar and mult_bar are both NULL");
    double *const g[KG_COUNT] = {gQ, gR, gHux, gq, gr, gA, gB, gd, gD2, gC, gc};
    if (std::all_of(g, g + KG_COUNT, [](double *x) { return x == nullptr; }))
        return lqrb_fail(h, -20, "every gradient output is NULL");
    if (gHux && hess_mode != LQRB_HESS_DENSE) return lqrb_fail(h, -22, "gHux needs LQRB_HESS_DENSE");
    if (gD2 && !D2) return lqrb_fail(h, -28, "gD2 needs an explicit D2");
    if (gC && z.sC == 0) return lqrb_fail(h, -29, "gC: p has no rows");
    if (gc && z.sc == 0) return lqrb_fail(h, -30, "gc: p has no rows");
    const int64_t K1 = N - 1;
    const int64_t per[KG_COUNT] = {(int64_t)n * n * N, (int64_t)m * m * K1, (int64_t)m * n * K1, (int64_t)n * N,
                                   (int64_t)m * K1,    (int64_t)n * n * K1, (int64_t)n * m * K1, (int64_t)n * K1,
                                   z.sD2,              z.sC,                z.sc};
    for (int o = 0; o < KG_COUNT; ++o)  // the kernel indexes an instance's elements in 31 bits
        if (g[o] && per[o] > (1ll << 30)) return lqrb_fail(h, -2, "n, m, N too large for the gradient kernel");
    if (batch == 0) return 0;
    LQRB_CUDA(h, cudaSetDevice(h->device));

    // inputs 0..10 in kkt_adjoint_data_map's source order, then the forward solution
    const std::vector<HostArray> inputs = {
        {Q, per[KG_Q] * 8},       {R, per[KG_R] * 8},           {Hux, Hux ? per[KG_HUX] * 8 : 0},
        {dz_bar, z.NN * 8},       {nullptr, 0},                 {A, per[KG_A] * 8},
        {B, per[KG_B] * 8},       {mult_bar, z.P * 8},          {D2, D2 ? z.sD2 * 8 : 0},
        {C, z.sC * 8},            {nullptr, 0},                 {dz, z.NN * 8},
        {mult, z.P * 8}};
    std::vector<HostArray> outputs;
    for (int o = 0; o < KG_COUNT; ++o) outputs.push_back({g[o], per[o] * 8});
    outputs.push_back({info, 4});
    KktGradTables tables;
    rc = kkt_grad_tables(h, s, &tables);
    if (rc) return rc;
    const std::string mkey = shape_key("kadj", s);
    auto mit = h->maps.find(mkey);
    const DevMap amap = mit != h->maps.end() ? mit->second : lqrb_get_map(h, mkey, kkt_adjoint_data_map(s));
    return lqrb_for_chunks(
        h, batch, 0, inputs, outputs, [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const int64_t ldb = lqrb_padded_batch(cb);
            double *data = (double *)lqrb_scratch(h, SCR_PACK_IN, (size_t)ldb * z.data_rows * 8, lane.index);
            double *dzp = (double *)lqrb_scratch(h, SCR_PACK_OUT, (size_t)ldb * z.NN * 8, lane.index);
            double *mp = (double *)lqrb_scratch(h, SCR_PACK_OUT2, (size_t)ldb * z.P * 8, lane.index);
            double *scr = (double *)lqrb_scratch(h, SCR_FACT, kkt_scratch_bytes(h, s, z, cb), lane.index);
            double *zh = (double *)lqrb_scratch(h, SCR_ADJOINT_Z, (size_t)cb * z.NN * 8, lane.index);
            double *mh = (double *)lqrb_scratch(h, SCR_ADJOINT_MULT, (size_t)cb * z.P * 8, lane.index);
            if (!data || !dzp || !mp || !scr || !zh || !mh) return 1000 + (int)cudaErrorMemoryAllocation;
            const int tile = lqrb_kkt_tile(h, n, m, N, p, hess_mode, s.d2x);
            int32_t rc = lqrb_gather_pack(h, amap, kkt_array_table(inputs, in), cb, tile, data, lane.stream);
            if (rc) return rc;
            KktRecord record;
            rc = kkt_solve_on(h, s, cb, 0, data, scr, dzp, mp, nullptr, (int32_t *)out[KG_COUNT], lane, &record);
            if (rc) return rc;
            rc = kkt_unpack_on(h, s, z, cb, dzp, mp, nullptr, zh, mh, nullptr, lane.stream);
            if (rc) return rc;
            KktGradArgs a = {};
            a.z = (const double *)in[11];
            a.mult = (const double *)in[12];
            a.zh = zh;
            a.multh = mh;
            a.t = tables;
            int64_t blocks = 0;
            for (int o = 0; o < KG_COUNT; ++o) {
                if (!out[o]) continue;
                a.kind[a.nout] = o;
                a.out[a.nout] = (double *)out[o];
                a.per[a.nout] = kkt_grad_div((uint32_t)per[o]);
                a.first_block[a.nout] = blocks;
                blocks += (cb * per[o] + KKT_GRAD_THREADS * KKT_GRAD_PER_THREAD - 1) / (KKT_GRAD_THREADS * KKT_GRAD_PER_THREAD);
                ++a.nout;
            }
            a.first_block[a.nout] = blocks;
            a.n = kkt_grad_div((uint32_t)n);
            a.m = kkt_grad_div((uint32_t)m);
            a.nn = kkt_grad_div((uint32_t)(n * n));
            a.mm = kkt_grad_div((uint32_t)(m * m));
            a.nm = kkt_grad_div((uint32_t)(n * m));
            a.NN = (int32_t)z.NN;
            a.P = (int32_t)z.P;
            a.diag = hess_mode == LQRB_HESS_DIAG;
            kkt_grad_kernel<<<(unsigned)blocks, KKT_GRAD_THREADS, 0, lane.stream>>>(a, n, m, N, cb);
            h->kernel_name += " + kkt_grad";
            LQRB_LAUNCH_CHECK(h, "kkt_grad_kernel");
            return 0;
        });
}


// ------------------------------------------------------------------ factor / solve split, dense extractors ----
// The reference keeps the Schur blocks (`shur_blocks`) and their Cholesky factor (`chol_blocks`) in the solver and
// runs the five steps of _solve! one by one (test/cholesky_solve.jl:14-35), re-using the factor for further
// right-hand sides.  Here the handle owns ONE kept factorisation (packed matrices + the block rows of U in the
// cooperative kernel's record layout, tile width 1); the fused kernels of lqrb_kkt_solve_f64 never touch it.

// row map of the right-hand-side array of phase 2: per knot g (w) | d (p2) | c (ps); sources 0 q, 1 r, 2 d, 3 c
static std::vector<RowMap> kkt_rhs_map(const KktShape &s) {
    std::vector<RowMap> map;
    int coff = 0;
    for (int k = 0; k < s.N; ++k) {
        const int mk = k < s.N - 1 ? s.m : 0, p2 = k < s.N - 1 ? s.n : 0, ps = s.p[k];
        for (int i = 0; i < s.n; ++i) map.push_back({0, k * s.n + i, 0.0});
        for (int i = 0; i < mk; ++i) map.push_back({1, k * s.m + i, 0.0});
        for (int i = 0; i < p2; ++i) map.push_back({2, k * s.n + i, 0.0});
        for (int i = 0; i < ps; ++i) map.push_back({3, coff + i, 0.0});
        coff += ps;
    }
    return map;
}

static std::string kept_key_of(const KktShape &s, int flags) {
    return shape_key("keep", s) + ((flags & LQRB_FLAG_SOC) ? "soc" : "");
}

extern "C" int32_t lqrb_kkt_factor_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                       const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                                       const double *R, const double *Hux, const double *A, const double *B,
                                       const double *D2, const double *C, int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!Q || !R || !A || !B) return lqrb_fail(h, -9, "a required input array is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, D2 != nullptr);
    const KktSizes z = kkt_sizes(s);
    if (z.sC > 0 && !C) return lqrb_fail(h, -15, "C is NULL but p has non-zero entries");
    h->kept_key.clear();
    h->kept_batch = 0;
    if (batch == 0) return 0;
    // sources in kkt_data_map order: Q R Hux q r A B d D2 C c — the right-hand-side rows are filled with zeros
    const double *src[11] = {Q, R, Hux, nullptr, nullptr, A, B, nullptr, D2, C, nullptr};
    const std::vector<HostArray> inputs = kkt_inputs(s, z, src);
    rc = lqrb_for_chunks(h, batch, batch, inputs, {{info, 4}},
                         [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
                             double *data = (double *)lqrb_scratch(h, SCR_KEEP_DATA, (size_t)cb * z.data_rows * 8);
                             double *rec = (double *)lqrb_scratch(h, SCR_KEEP_REC, (size_t)cb * z.rec_rows * 8);
                             if (!data || !rec) return 1000 + (int)cudaErrorMemoryAllocation;
                             const ArrayTable t = kkt_array_table(inputs, in);
                             int32_t rc = lqrb_gather_pack(h, lqrb_get_map(h, shape_key("kd", s), kkt_data_map(s)), t,
                                                           cb, 1, data, lane.stream);
                             if (rc) return rc;
                             KktCoopExtra ex;
                             ex.phase = 1;
                             return launch_kkt_coop(h, n, m, N, p, hess_mode, s.d2x, flags, cb, data, rec, nullptr,
                                                    nullptr, nullptr, (int32_t *)out[0], lane, &ex);
                         });
    if (rc) return rc;
    h->kept_key = kept_key_of(s, flags);
    h->kept_batch = batch;
    return 0;
}

extern "C" int32_t lqrb_kkt_solve_factored_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                               const int32_t *p, int32_t hess_mode, int32_t explicit_d2,
                                               int32_t flags, const double *q, const double *r, const double *d,
                                               const double *c, double *dz, double *mult, double *res,
                                               int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    const bool soc = (flags & LQRB_FLAG_SOC) != 0;
    if (!soc && (!q || !r)) return lqrb_fail(h, -10, "q / r is NULL");
    if (!d) return lqrb_fail(h, -12, "d is NULL");
    if (!dz) return lqrb_fail(h, -14, "dz is NULL");
    if (!mult) return lqrb_fail(h, -15, "mult is NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, explicit_d2);
    const KktSizes z = kkt_sizes(s);
    if (z.sc > 0 && !c) return lqrb_fail(h, -13, "c is NULL but p has non-zero entries");
    if (h->kept_key.empty() || h->kept_key != kept_key_of(s, flags) || h->kept_batch != batch)
        return lqrb_fail(h, -1, "no kept factorisation of this shape / batch / flags: call lqrb_kkt_factor_f64 first");
    if (batch == 0) return 0;
    const std::vector<HostArray> inputs = {
        {q, (int64_t)n * N * 8}, {r, (int64_t)m * (N - 1) * 8}, {d, (int64_t)n * (N - 1) * 8}, {c, z.sc * 8}};
    return lqrb_for_chunks(
        h, batch, batch, inputs, {{dz, z.NN * 8}, {mult, z.P * 8}, {res, z.NN * 8}, {info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            double *rhs = (double *)lqrb_scratch(h, SCR_PACK_IN2, (size_t)cb * (z.NN + z.P) * 8, lane.index);
            if (!rhs) return 1000 + (int)cudaErrorMemoryAllocation;
            const ArrayTable t = kkt_array_table(inputs, in);
            int32_t rc = lqrb_gather_pack(h, lqrb_get_map(h, shape_key("krhs", s), kkt_rhs_map(s)), t, cb, 1, rhs,
                                          lane.stream);
            if (rc) return rc;
            // tile width 1: the packed outputs ARE the instance-major arrays
            KktCoopExtra ex;
            ex.phase = 2;
            ex.rhs = rhs;
            return launch_kkt_coop(h, n, m, N, p, hess_mode, s.d2x, flags, cb, (const double *)h->scratch[SCR_KEEP_DATA][0],
                                   (double *)h->scratch[SCR_KEEP_REC][0], (double *)out[0], (double *)out[1],
                                   (double *)out[2], (int32_t *)out[3], lane, &ex);
        });
}

// dense P x P image of the block rows (copy_shur_factors! / copy_block!, src/jacobian_blocks.jl:173-211):
// knot k contributes A (lam_{k-1}, aliasing C_{k-1}), B (mu_k), D, E, F; the vector slots give h (c_k, d_{k-1}).
static void assemble_block_rows(const KktShape &s, const double *rec, int64_t P, bool factor, double *M, double *hv) {
    const int n = s.n, N = s.N;
    int64_t off = 0;  // mult offset of mu_k
    for (int k = 0; k < N; ++k) {
        const int p1 = k > 0 ? n : 0, ps = s.p[k], p2 = k < N - 1 ? n : 0;
        const double *rB = rec, *rD = rB + (int64_t)ps * ps, *rE = rD + (int64_t)p1 * ps, *rF = rE + (int64_t)ps * p2,
                     *rmu = rF + (int64_t)p1 * p2, *rC = rmu + ps, *rl = rC + (int64_t)p1 * p1;
        const int64_t i1 = off - p1, is = off, i2 = off + ps;
        auto put = [&](int64_t i, int64_t j, double v) {
            M[i + j * P] = v;
            if (!factor) M[j + i * P] = v;  // Symmetric(S, :U)
        };
        for (int j = 0; j < p1; ++j)
            for (int i = 0; i <= j; ++i) put(i1 + i, i1 + j, rC[i + (int64_t)j * p1]);
        for (int j = 0; j < ps; ++j)
            for (int i = 0; i <= j; ++i) put(is + i, is + j, rB[i + (int64_t)j * ps]);
        for (int j = 0; j < ps; ++j)
            for (int i = 0; i < p1; ++i) put(i1 + i, is + j, rD[i + (int64_t)j * p1]);
        for (int j = 0; j < p2; ++j)
            for (int i = 0; i < ps; ++i) put(is + i, i2 + j, rE[i + (int64_t)j * ps]);
        for (int j = 0; j < p2; ++j)
            for (int i = 0; i < p1; ++i) put(i1 + i, i2 + j, rF[i + (int64_t)j * p1]);
        if (hv) {
            for (int i = 0; i < ps; ++i) hv[is + i] = rmu[i];
            for (int i = 0; i < p1; ++i) hv[i1 + i] = rl[i];
        }
        rec += kkt_coop_rec_knot_rows(p1, ps, p2);
        off += ps + p2;
    }
}

extern "C" int32_t lqrb_kkt_get_shur_f64(lqrb_handle_t h, int32_t n, int32_t m, int32_t N, int64_t batch,
                                         const int32_t *p, int32_t hess_mode, int32_t flags, const double *Q,
                                         const double *R, const double *Hux, const double *q, const double *r,
                                         const double *A, const double *B, const double *d, const double *D2,
                                         const double *C, const double *c, double *S, double *hvec, double *U,
                                         int32_t *info) {
    int32_t rc = check_kkt(h, n, m, N, batch, p, hess_mode);
    if (rc) return rc;
    if (!Q || !R || !q || !r || !A || !B || !d) return lqrb_fail(h, -9, "a required input array is NULL");
    if (!S && !hvec && !U) return lqrb_fail(h, -20, "S, h and U are all NULL");
    LQRB_CUDA(h, cudaSetDevice(h->device));
    const KktShape s = make_shape(n, m, N, p, hess_mode, D2 != nullptr);
    const KktSizes z = kkt_sizes(s);
    if (z.sC > 0 && (!C || !c)) return lqrb_fail(h, -18, "C/c is NULL but p has non-zero entries");
    if (batch == 0) return 0;
    const double *src[11] = {Q, R, Hux, q, r, A, B, d, D2, C, c};
    const std::vector<HostArray> inputs = kkt_inputs(s, z, src);
    // S, h and U are assembled on the host and written with cudaMemcpyDefault, whatever memory they are in
    return lqrb_for_chunks(
        h, batch, batch, inputs, {{info, 4}},
        [&](Lane lane, int64_t cb, const void *const *in, void *const *out) -> int32_t {
            const cudaStream_t st = lane.stream;
            double *data = (double *)lqrb_scratch(h, SCR_PACK_IN, (size_t)cb * z.data_rows * 8, lane.index);
            double *rec = (double *)lqrb_scratch(h, SCR_FACT, (size_t)cb * z.rec_rows * 8, lane.index);
            double *sd = (double *)lqrb_scratch(h, SCR_PACK_OUT, (size_t)cb * z.rec_rows * 8, lane.index);
            double *sol = (double *)lqrb_scratch(h, SCR_PACK_OUT2, (size_t)cb * (z.NN + z.P) * 8, lane.index);
            if (!data || !rec || !sd || !sol) return 1000 + (int)cudaErrorMemoryAllocation;
            const ArrayTable t = kkt_array_table(inputs, in);
            int32_t rc = lqrb_gather_pack(h, lqrb_get_map(h, shape_key("kd", s), kkt_data_map(s)), t, cb, 1, data, st);
            if (rc) return rc;
            LQRB_CUDA(h, cudaMemsetAsync(sd, 0, (size_t)cb * z.rec_rows * 8, st));
            KktCoopExtra ex;
            ex.phase = 0;
            ex.sdump = sd;
            rc = launch_kkt_coop(h, n, m, N, p, hess_mode, s.d2x, flags, cb, data, rec, sol, sol + cb * z.NN, nullptr,
                                 (int32_t *)out[0], lane, &ex);
            if (rc) return rc;
            std::vector<double> hrec((size_t)z.rec_rows), hsd((size_t)z.rec_rows), dense((size_t)z.P * z.P), hv((size_t)z.P);
            for (int64_t i = 0; i < cb; ++i) {
                LQRB_CUDA(h, cudaMemcpyAsync(hrec.data(), rec + i * z.rec_rows, (size_t)z.rec_rows * 8, cudaMemcpyDeviceToHost, st));
                LQRB_CUDA(h, cudaMemcpyAsync(hsd.data(), sd + i * z.rec_rows, (size_t)z.rec_rows * 8, cudaMemcpyDeviceToHost, st));
                LQRB_CUDA(h, cudaStreamSynchronize(st));
                if (S || hvec) {
                    std::fill(dense.begin(), dense.end(), 0.0);
                    assemble_block_rows(s, hsd.data(), z.P, false, dense.data(), hv.data());
                    if (S) LQRB_CUDA(h, cudaMemcpy(S + i * z.P * z.P, dense.data(), (size_t)z.P * z.P * 8, cudaMemcpyDefault));
                    if (hvec) LQRB_CUDA(h, cudaMemcpy(hvec + i * z.P, hv.data(), (size_t)z.P * 8, cudaMemcpyDefault));
                }
                if (U) {
                    std::fill(dense.begin(), dense.end(), 0.0);
                    assemble_block_rows(s, hrec.data(), z.P, true, dense.data(), nullptr);
                    LQRB_CUDA(h, cudaMemcpy(U + i * z.P * z.P, dense.data(), (size_t)z.P * z.P * 8, cudaMemcpyDefault));
                }
            }
            return 0;
        });
}

extern "C" int32_t lqrb_kkt_last_condition(lqrb_handle_t h, int64_t count, int32_t *log2_pivot_ratio, int64_t *resolved) {
    if (!h) return -1;
    if (count < 0) return -2;
    if (log2_pivot_ratio) {
        for (int64_t i = 0; i < count; ++i)
            log2_pivot_ratio[i] = i < (int64_t)h->last_cond.size() ? h->last_cond[(size_t)i] : -1;
    }
    if (resolved) *resolved = h->last_refined;
    return 0;
}
