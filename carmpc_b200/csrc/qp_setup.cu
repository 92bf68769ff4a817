// Host-side setup of the batched QP solver: equilibration, the shared KKT inverse, structure analysis (independent
// chains, causal row extents), tiling tables and the float64 polish matrices.  Runs once per controller.
//
// The matrices it consumes are the reference's own: H, h from lib/matrix_gen.py:35-72 and the constraint stacks of
// lib/mpc.py:196-253 multiplied into S and T (lib/mpc.py:319-332); see carmpc_b200/condensed.py.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <numeric>

#include "qp_internal.cuh"

namespace carmpc {

namespace {

inline int round4(int x) { return (x + 3) & ~3; }
inline int floor4(int x) { return x & ~3; }

// in-place Cholesky A = L L' (lower), row-major n x n.  Returns false when not positive definite.
bool cholesky(std::vector<double>& A, int n) {
    for (int j = 0; j < n; ++j) {
        double d = A[j * n + j];
        for (int k = 0; k < j; ++k) d -= A[j * n + k] * A[j * n + k];
        if (!(d > 0.0)) return false;
        d = sqrt(d);
        A[j * n + j] = d;
        for (int i = j + 1; i < n; ++i) {
            double s = A[i * n + j];
            for (int k = 0; k < j; ++k) s -= A[i * n + k] * A[j * n + k];
            A[i * n + j] = s / d;
        }
    }
    return true;
}

// inverse of an SPD matrix through its Cholesky factor
bool spd_inverse(const std::vector<double>& A, int n, std::vector<double>& inv) {
    std::vector<double> L(A);
    if (!cholesky(L, n)) return false;
    inv.assign((size_t)n * n, 0.0);
    std::vector<double> y(n);
    for (int c = 0; c < n; ++c) {
        for (int i = 0; i < n; ++i) {                   // L y = e_c
            double s = (i == c) ? 1.0 : 0.0;
            for (int k = 0; k < i; ++k) s -= L[i * n + k] * y[k];
            y[i] = s / L[i * n + i];
        }
        for (int i = n - 1; i >= 0; --i) {              // L' x = y
            double s = y[i];
            for (int k = i + 1; k < n; ++k) s -= L[k * n + i] * inv[(size_t)k * n + c];
            inv[(size_t)i * n + c] = s / L[i * n + i];
        }
    }
    for (int i = 0; i < n; ++i)                          // symmetrise
        for (int j = i + 1; j < n; ++j) {
            const double v = 0.5 * (inv[(size_t)i * n + j] + inv[(size_t)j * n + i]);
            inv[(size_t)i * n + j] = inv[(size_t)j * n + i] = v;
        }
    return true;
}

// Modified Ruiz equilibration of [[H, A'], [A, 0]] with A = [G; I] (OSQP's scaling; tools/admm_model.py mirrors it)
void ruiz(const std::vector<double>& H, const std::vector<double>& G, int n, int m, int iters, std::vector<double>& D,
          std::vector<double>& Eg, std::vector<double>& Eb, double& c) {
    D.assign(n, 1.0);
    Eg.assign(m, 1.0);
    Eb.assign(n, 1.0);
    c = 1.0;
    std::vector<double> col(n), rowg(m), rowb(n);
    for (int it = 0; it < iters; ++it) {
        for (int j = 0; j < n; ++j) {
            double mx = 0;
            for (int i = 0; i < n; ++i) mx = std::max(mx, fabs(c * D[i] * H[(size_t)i * n + j] * D[j]));
            for (int i = 0; i < m; ++i) mx = std::max(mx, fabs(Eg[i] * G[(size_t)i * n + j] * D[j]));
            mx = std::max(mx, fabs(Eb[j] * D[j]));
            col[j] = mx < 1e-4 ? 1.0 : mx;
        }
        for (int i = 0; i < m; ++i) {
            double mx = 0;
            for (int j = 0; j < n; ++j) mx = std::max(mx, fabs(Eg[i] * G[(size_t)i * n + j] * D[j]));
            rowg[i] = mx < 1e-4 ? 1.0 : mx;
        }
        for (int j = 0; j < n; ++j) {
            const double v = fabs(Eb[j] * D[j]);
            rowb[j] = v < 1e-4 ? 1.0 : v;
        }
        for (int j = 0; j < n; ++j) D[j] /= sqrt(col[j]);
        for (int i = 0; i < m; ++i) Eg[i] /= sqrt(rowg[i]);
        for (int j = 0; j < n; ++j) Eb[j] /= sqrt(rowb[j]);
        double avg = 0;
        for (int j = 0; j < n; ++j) {
            double mx = 0;
            for (int i = 0; i < n; ++i) mx = std::max(mx, fabs(c * D[i] * H[(size_t)i * n + j] * D[j]));
            avg += mx;
        }
        avg /= n;
        if (avg > 1e-4) c /= avg;
    }
}

struct UnionFind {
    std::vector<int> p;
    explicit UnionFind(int n) : p(n) { std::iota(p.begin(), p.end(), 0); }
    int find(int x) { while (p[x] != x) x = p[x] = p[p[x]]; return x; }
    void unite(int a, int b) { a = find(a); b = find(b); if (a != b) p[std::max(a, b)] = std::min(a, b); }
};

}  // namespace

size_t admm_smem_bytes(const QPHost& h, int S, bool mats) {
    const AdmmTables& g = h.geo;
    const int Bt = 32 * S;
    size_t b = 0;
    b += sizeof(float) * (size_t)g.ktot * Bt;            // V
    b += sizeof(float) * (size_t)g.npad4 * Bt;           // x~
    b += sizeof(float) * (size_t)g.m_phys * Bt;          // hi
    if (mats) b += sizeof(float) * ((size_t)g.nA_rows * g.ktot + (size_t)g.m_phys * g.npad4);
    b += sizeof(float) * ((size_t)g.m_phys + 3 * (size_t)g.nA_rows);     // width, lam, lbs, ubs
    b += sizeof(int) * (2 * (size_t)g.m_phys + (size_t)g.nA_rows);          // vpos, row_id, var_id
    b += sizeof(float) * (2 * (size_t)g.m_phys + 4 * (size_t)g.nA_rows);     // scales for checks / outputs
    b += sizeof(double) * (6 * (size_t)g.m_phys + 4 * (size_t)g.nA_rows);    // his, Gxs, Gcs, KF
    b += 16 * 20;                                        // alignment slack of the carve-up
    b += sizeof(int4) * (size_t)g.nGA + sizeof(int2) * (size_t)g.nGB;
    b += (sizeof(double) * 5 + sizeof(int) * 5 + sizeof(float) * 5) * (size_t)Bt;   // per-slot state
    b += 256;
    return b;
}

int qp_host_setup(int n, int m_in, int kpre, const double* H_in, const double* F_in, const double* G_in,
                  const double* Gx_in, const double* Gc_in, const double* lo_in, const double* hi_in,
                  const double* lb_in, const double* ub_in, const double* Px_in, const double* Pc_in,
                  const double* pre_lo_in, const double* pre_hi_in, const carmpc_qp_opts& opts, QPHost* out) {
    QPHost& q = *out;
    q.n = n;
    q.m = m_in;
    q.kpre = kpre;
    q.opts = opts;
    const int m = m_in, mt = m + n;
    const double rho = opts.rho;

    // ---- logical copies; rows bounded only from below are negated so that every live row has a finite hi ----------
    q.H.assign(H_in, H_in + (size_t)n * n);
    q.F.assign(F_in, F_in + (size_t)n * 4);
    q.G.assign(G_in, G_in + (size_t)m * n);
    q.Gx.assign(Gx_in, Gx_in + (size_t)m * 4);
    q.Gc.assign((size_t)m, 0.0);
    if (Gc_in) q.Gc.assign(Gc_in, Gc_in + m);
    q.hi.assign(mt, 0.0);
    q.lo.assign(mt, 0.0);
    q.rsign.assign((size_t)m, 1.0);
    std::vector<char> live(m, 1);
    for (int i = 0; i < m; ++i) {
        double lo = lo_in[i], hi = hi_in[i];
        if (isnan(lo) || isnan(hi)) { set_error("carmpc_qp_create: NaN bound in row %d", i); return CARMPC_ERR_INVALID; }
        if (isinf(hi) && hi > 0 && isinf(lo) && lo < 0) live[i] = 0;
        else if (isinf(hi) && hi > 0) {
            for (int j = 0; j < n; ++j) q.G[(size_t)i * n + j] = -q.G[(size_t)i * n + j];
            for (int c = 0; c < 4; ++c) q.Gx[(size_t)i * 4 + c] = -q.Gx[(size_t)i * 4 + c];
            q.Gc[i] = -q.Gc[i];
            q.rsign[i] = -1.0;
            const double t = hi; hi = -lo; lo = -t;
        }
        q.hi[i] = hi;
        q.lo[i] = lo;
    }
    for (int j = 0; j < n; ++j) { q.hi[m + j] = ub_in[j]; q.lo[m + j] = lb_in[j]; }
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j)
            if (!isfinite(q.H[(size_t)i * n + j])) { set_error("carmpc_qp_create: non-finite H"); return CARMPC_ERR_INVALID; }

    // ---- equilibration ---------------------------------------------------------------------------------------------------
    ruiz(q.H, q.G, n, m, opts.scaling_iters, q.D, q.Eg, q.Eb, q.cscale);
    const std::vector<double>&D = q.D, &Eg = q.Eg, &Eb = q.Eb;
    const double cs = q.cscale;
    std::vector<double> Hs((size_t)n * n), K((size_t)n * n), lam(n);
    q.Gs64.assign((size_t)m * n, 0.0);
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < n; ++j) Hs[(size_t)i * n + j] = cs * D[i] * q.H[(size_t)i * n + j] * D[j];
    for (int i = 0; i < m; ++i)
        for (int j = 0; j < n; ++j) q.Gs64[(size_t)i * n + j] = live[i] ? Eg[i] * q.G[(size_t)i * n + j] * D[j] : 0.0;
    // Entries below 1e-12 of their row's largest are rounding noise of the constraint stacks (e.g. 1e-16 coefficients
    // in the shipped terminal sets): drop them so that the chain structure is exact.  The float32 ADMM only has to
    // find the active set; the polish works on the untouched G.
    for (int i = 0; i < m; ++i) {
        double mx = 0;
        for (int j = 0; j < n; ++j) mx = std::max(mx, fabs(q.Gs64[(size_t)i * n + j]));
        for (int j = 0; j < n; ++j)
            if (fabs(q.Gs64[(size_t)i * n + j]) <= 1e-12 * mx) q.Gs64[(size_t)i * n + j] = 0.0;
    }
    for (int j = 0; j < n; ++j) lam[j] = Eb[j] * D[j];
    K = Hs;
    for (int i = 0; i < m; ++i) {
        const double* g = &q.Gs64[(size_t)i * n];
        for (int a = 0; a < n; ++a) {
            if (g[a] == 0.0) continue;
            const double ga = rho * g[a];
            for (int b = 0; b < n; ++b) K[(size_t)a * n + b] += ga * g[b];
        }
    }
    for (int j = 0; j < n; ++j) K[(size_t)j * n + j] += rho * lam[j] * lam[j];
    if (!spd_inverse(K, n, q.Kinv)) { set_error("carmpc_qp_create: H + rho A'A is not positive definite"); return CARMPC_ERR_NUMERIC; }
    if (!spd_inverse(q.H, n, q.Hinv)) { set_error("carmpc_qp_create: H is not positive definite"); return CARMPC_ERR_NUMERIC; }

    // ---- structure: independent chains (connected components of variables) ------------------------------------------------
    UnionFind uf(n);
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j)
            if (fabs(Hs[(size_t)i * n + j]) > 1e-9 * sqrt(fabs(Hs[(size_t)i * n + i] * Hs[(size_t)j * n + j]))) uf.unite(i, j);
    std::vector<std::vector<int>> row_vars(m);
    for (int i = 0; i < m; ++i) {
        if (!live[i]) continue;
        double mx = 0;
        for (int j = 0; j < n; ++j) mx = std::max(mx, fabs(q.Gs64[(size_t)i * n + j]));
        for (int j = 0; j < n; ++j)
            if (q.Gs64[(size_t)i * n + j] != 0.0 && mx > 0) row_vars[i].push_back(j);
        for (size_t t = 1; t < row_vars[i].size(); ++t) uf.unite(row_vars[i][0], row_vars[i][t]);
    }
    std::vector<int> comp(n), comp_label(n, -1);
    int ncomp = 0;
    for (int j = 0; j < n; ++j) {
        const int r = uf.find(j);
        if (comp_label[r] < 0) comp_label[r] = ncomp++;
        comp[j] = comp_label[r];
    }
    std::vector<int> perm(n), pos(n);                    // perm[p] = logical variable at permuted position p
    std::iota(perm.begin(), perm.end(), 0);
    std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return comp[a] < comp[b]; });
    for (int p = 0; p < n; ++p) pos[perm[p]] = p;

    // ---- size class ----------------------------------------------------------------------------------------------------------
    std::vector<int> rows;                                // live general rows
    for (int i = 0; i < m; ++i) if (live[i]) rows.push_back(i);
    const int mv = (int)rows.size();
    const int nGA = (n + kRA - 1) / kRA;
    int S, GA, GB;
    if (nGA <= 8 && mv <= 2 * 8 * kRB) { S = 4; GA = 1; GB = 2; }
    else if (nGA <= 16 && mv <= 4 * 8 * kRB) { S = 2; GA = 2; GB = 4; }
    else if (nGA <= 32 && mv <= 7 * 8 * kRB) { S = 1; GA = 4; GB = 7; }
    else { set_error("carmpc_qp_create: problem too large (n <= %d, general rows <= %d)", kMaxN, kMaxM); return CARMPC_ERR_UNSUPPORTED; }
    q.samples_per_lane = S;
    q.ga_per_warp = GA;
    q.gb_per_warp = GB;

    AdmmTables& g = q.geo;
    memset(&g, 0, sizeof(g));
    g.n = n; g.m = m; g.mt = mt; g.kpre = kpre;
    g.nA_rows = nGA * kRA;
    g.nGA = nGA;
    g.nGB = GB * kAdmmWarps;
    g.m_phys = g.nGB * kRB;
    g.npad4 = round4(g.nA_rows);
    g.mv4 = round4(mv);
    g.ktot = g.mv4 + g.npad4;
    g.rho = (float)rho; g.alpha = (float)opts.alpha; g.eps_abs = (float)opts.eps_abs; g.eps_rel = (float)opts.eps_rel;
    g.eps_inf = (float)opts.eps_prim_inf; g.check_every = opts.check_every;

    // ---- V order of the general rows: by chain, so that each chain's rows are one contiguous K range ------------------------
    std::vector<int> row_comp(m, 0), row_beg(m, 0), row_end(m, 0);
    for (int i : rows) {
        int b = n, e = 0;
        for (int j : row_vars[i]) { b = std::min(b, pos[j]); e = std::max(e, pos[j] + 1); }
        if (row_vars[i].empty()) { b = 0; e = 0; }
        row_comp[i] = row_vars[i].empty() ? 0 : comp[row_vars[i][0]];
        row_beg[i] = b; row_end[i] = e;
    }
    std::vector<int> vorder(rows);
    std::stable_sort(vorder.begin(), vorder.end(), [&](int a, int b) {
        if (row_comp[a] != row_comp[b]) return row_comp[a] < row_comp[b];
        return row_end[a] < row_end[b];
    });
    std::vector<int> vpos_of(m, -1);
    for (int p = 0; p < mv; ++p) vpos_of[vorder[p]] = p;

    // ---- owner (physical) order: groups of kRB rows with similar extents, spread over the warps by cost (LPT) ---------------
    const int nLG = (mv + kRB - 1) / kRB;
    std::vector<int> lg_cost(nLG), lg_order(nLG);
    for (int lg = 0; lg < nLG; ++lg) {
        int b = n, e = 0;
        for (int r = lg * kRB; r < std::min(mv, (lg + 1) * kRB); ++r) { b = std::min(b, row_beg[vorder[r]]); e = std::max(e, row_end[vorder[r]]); }
        lg_cost[lg] = std::max(0, round4(e) - floor4(std::min(b, e)));
    }
    std::iota(lg_order.begin(), lg_order.end(), 0);
    std::stable_sort(lg_order.begin(), lg_order.end(), [&](int a, int b) { return lg_cost[a] > lg_cost[b]; });
    std::vector<int> warp_load(kAdmmWarps, 0), warp_used(kAdmmWarps, 0), phys_of_lg(nLG, -1);
    for (int lg : lg_order) {
        int best = -1;
        for (int w = 0; w < kAdmmWarps; ++w)
            if (warp_used[w] < GB && (best < 0 || warp_load[w] < warp_load[best])) best = w;
        phys_of_lg[lg] = warp_used[best] * kAdmmWarps + best;
        warp_used[best]++;
        warp_load[best] += lg_cost[lg];
    }

    // ---- padded device images ---------------------------------------------------------------------------------------------------
    q.Gs.assign((size_t)g.m_phys * g.npad4, 0.f);
    q.his.assign(g.m_phys, 3.0e38);
    q.Gxs.assign((size_t)g.m_phys * 4, 0.0);
    q.Gcs.assign(g.m_phys, 0.0);
    q.width.assign(g.m_phys, INFINITY);
    q.Einv_g.assign(g.m_phys, 0.f);
    q.Esc_g.assign(g.m_phys, 0.f);
    q.vpos.assign(g.m_phys, 0);
    q.row_id.assign(g.m_phys, -1);
    q.segB.assign(g.nGB, make_int2(0, 0));
    // pad rows park their (always zero) V entry on a pad slot when there is one, else on their own group's first row
    const int park = mv < g.mv4 ? mv : -1;
    double flopsB = 0;
    for (int lg = 0; lg < nLG; ++lg) {
        const int pg = phys_of_lg[lg];
        int b = n, e = 0;
        for (int r = 0; r < kRB; ++r) {
            const int src = lg * kRB + r;
            const int pi = pg * kRB + r;
            if (src >= mv) continue;
            const int i = vorder[src];
            for (int j = 0; j < n; ++j) q.Gs[(size_t)pi * g.npad4 + pos[j]] = (float)q.Gs64[(size_t)i * n + j];
            q.his[pi] = Eg[i] * q.hi[i];
            for (int c = 0; c < 4; ++c) q.Gxs[(size_t)pi * 4 + c] = Eg[i] * q.Gx[(size_t)i * 4 + c];
            q.Gcs[pi] = Eg[i] * q.Gc[i];
            q.width[pi] = isinf(q.lo[i]) ? INFINITY : (float)(Eg[i] * (q.hi[i] - q.lo[i]));
            q.Einv_g[pi] = (float)(1.0 / Eg[i]);
            q.Esc_g[pi] = (float)Eg[i];
            q.vpos[pi] = vpos_of[i];
            q.row_id[pi] = i;
            b = std::min(b, row_beg[i]); e = std::max(e, row_end[i]);
        }
        if (e > b) { q.segB[pg] = make_int2(floor4(b), round4(e)); flopsB += 2.0 * kRB * (round4(e) - floor4(b)); }
    }
    for (int pi = 0; pi < g.m_phys; ++pi)
        if (q.row_id[pi] < 0) q.vpos[pi] = park >= 0 ? park : -1;          // -1: the kernel skips the store

    // variables
    q.lam.assign(g.nA_rows, 0.f); q.lbs.assign(g.nA_rows, -INFINITY); q.ubs.assign(g.nA_rows, INFINITY);
    q.Einv_b.assign(g.nA_rows, 0.f); q.Esc_b.assign(g.nA_rows, 0.f); q.Dinv.assign(g.nA_rows, 0.f); q.Dsc.assign(g.nA_rows, 0.f);
    q.KF.assign((size_t)g.nA_rows * 4, 0.0);
    q.var_id.assign(g.nA_rows, -1);
    for (int p = 0; p < n; ++p) {
        const int j = perm[p];
        q.lam[p] = (float)lam[j];
        q.lbs[p] = isinf(lb_in[j]) ? -INFINITY : (float)(Eb[j] * lb_in[j]);
        q.ubs[p] = isinf(ub_in[j]) ? INFINITY : (float)(Eb[j] * ub_in[j]);
        q.Einv_b[p] = (float)(1.0 / Eb[j]);
        q.Esc_b[p] = (float)Eb[j];
        q.Dinv[p] = (float)(1.0 / D[j]);
        q.Dsc[p] = (float)D[j];
        q.var_id[p] = j;
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int k = 0; k < n; ++k) s += q.Kinv[(size_t)j * n + k] * cs * D[k] * q.F[(size_t)k * 4 + c];
            q.KF[(size_t)p * 4 + c] = -s;
        }
    }

    // P = rho K^-1 [Gs' | diag(lam)] in V order, GsT in V order; structural zeros between chains made exact
    q.P.assign((size_t)g.nA_rows * g.ktot, 0.f);
    q.GsT.assign((size_t)g.nA_rows * g.mv4, 0.f);
    std::vector<double> KG((size_t)n * m, 0.0);            // K^-1 Gs'
    for (int a = 0; a < n; ++a)
        for (int i : rows) {
            double s = 0;
            const double* gi = &q.Gs64[(size_t)i * n];
            for (int k = 0; k < n; ++k) s += q.Kinv[(size_t)a * n + k] * gi[k];
            KG[(size_t)a * m + i] = s;
        }
    for (int p = 0; p < n; ++p) {
        const int j = perm[p];
        for (int i : rows) {
            if (row_vars[i].empty() || row_comp[i] != comp[j]) continue;
            q.P[(size_t)p * g.ktot + vpos_of[i]] = (float)(rho * KG[(size_t)j * m + i]);
            q.GsT[(size_t)p * g.mv4 + vpos_of[i]] = (float)q.Gs64[(size_t)i * n + j];
        }
        for (int p2 = 0; p2 < n; ++p2) {
            const int j2 = perm[p2];
            if (comp[j2] != comp[j]) continue;
            q.P[(size_t)p * g.ktot + g.mv4 + p2] = (float)(rho * q.Kinv[(size_t)j * n + j2] * lam[j2]);
        }
    }
    // stage-A segments per group of kRA permuted variables
    q.segA.assign(g.nGA, make_int4(0, 0, 0, 0));
    double flopsA = 0;
    for (int ga = 0; ga < g.nGA; ++ga) {
        int gb = mv, ge = 0, bb = n, be = 0;
        for (int p = ga * kRA; p < std::min(n, (ga + 1) * kRA); ++p) {
            const int c = comp[perm[p]];
            for (int i : rows) if (!row_vars[i].empty() && row_comp[i] == c) { gb = std::min(gb, vpos_of[i]); ge = std::max(ge, vpos_of[i] + 1); }
            for (int p2 = 0; p2 < n; ++p2) if (comp[perm[p2]] == c) { bb = std::min(bb, p2); be = std::max(be, p2 + 1); }
        }
        if (ge < gb) { gb = 0; ge = 0; }
        if (be < bb) { bb = 0; be = 0; }
        q.segA[ga] = make_int4(floor4(gb), round4(ge), g.mv4 + floor4(bb), g.mv4 + round4(be));
        flopsA += 2.0 * kRA * ((round4(ge) - floor4(gb)) + (round4(be) - floor4(bb)));
    }
    q.flops_per_iter = flopsA + flopsB;
    q.flops_per_iter_dense = 2.0 * n * (double)(mv + n) + 2.0 * (double)mv * n;

    // pre-check rows
    q.Px.assign(Px_in ? Px_in : nullptr, Px_in ? Px_in + (size_t)kpre * 4 : nullptr);
    q.Pc.assign((size_t)kpre, 0.0);
    if (Pc_in) q.Pc.assign(Pc_in, Pc_in + kpre);
    q.pre_lo.assign(pre_lo_in ? pre_lo_in : nullptr, pre_lo_in ? pre_lo_in + kpre : nullptr);
    q.pre_hi.assign(pre_hi_in ? pre_hi_in : nullptr, pre_hi_in ? pre_hi_in + kpre : nullptr);

    // ---- polish matrices (logical order, unscaled, float64) ---------------------------------------------------------------------------
    q.AH.assign((size_t)mt * n, 0.0);
    for (int i = 0; i < m; ++i) {
        if (!live[i]) continue;
        for (int b = 0; b < n; ++b) {
            double s = 0;
            for (int k = 0; k < n; ++k) s += q.G[(size_t)i * n + k] * q.Hinv[(size_t)k * n + b];
            q.AH[(size_t)i * n + b] = s;
        }
    }
    for (int j = 0; j < n; ++j)
        for (int b = 0; b < n; ++b) q.AH[(size_t)(m + j) * n + b] = q.Hinv[(size_t)j * n + b];
    q.AHA.assign((size_t)mt * mt, 0.0);
    for (int a = 0; a < mt; ++a) {
        const double* ah = &q.AH[(size_t)a * n];
        for (int b = 0; b < m; ++b) {
            if (!live[b]) continue;
            double s = 0;
            const double* gb = &q.G[(size_t)b * n];
            for (int k = 0; k < n; ++k) s += ah[k] * gb[k];
            q.AHA[(size_t)a * mt + b] = s;
        }
        for (int j = 0; j < n; ++j) q.AHA[(size_t)a * mt + m + j] = ah[j];
    }
    for (int i = 0; i < m; ++i)
        if (!live[i]) { q.hi[i] = INFINITY; q.lo[i] = -INFINITY; }
    q.Uu.assign((size_t)n * 4, 0.0);
    for (int j = 0; j < n; ++j)
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            for (int k = 0; k < n; ++k) s += q.Hinv[(size_t)j * n + k] * q.F[(size_t)k * 4 + c];
            q.Uu[(size_t)j * 4 + c] = -s;
        }
    q.AUu.assign((size_t)mt * 4, 0.0);
    for (int i = 0; i < mt; ++i)
        for (int c = 0; c < 4; ++c) {
            double s = 0;
            if (i < m) { if (live[i]) for (int k = 0; k < n; ++k) s += q.G[(size_t)i * n + k] * q.Uu[(size_t)k * 4 + c]; }
            else s = q.Uu[(size_t)(i - m) * 4 + c];
            q.AUu[(size_t)i * 4 + c] = s;
        }

    // ---- tensor-core form (qp_admm_tc.cu): logical order, B operands as swizzled TF32 hi / lo chunk images ---------------------
    // One part for the whole problem when it fits tensor memory; else (horizon 80) one part per independent chain of the
    // variable graph - K is block diagonal over the chains, so the ADMM iteration of the whole problem IS the chains'
    // iterations side by side, and each chain is a horizon-40-sized problem.
    auto build_part = [&](const std::vector<int>& vars, const std::vector<int>& prows, TcPart& P) {
        TcTables& t = P.t;
        memset(&t, 0, sizeof(t));
        const int nv = (int)vars.size(), nr = (int)prows.size();
        const int np = std::max(16, (nv + 15) / 16 * 16), mp = std::max(16, (nr + 15) / 16 * 16);
        t.n = n; t.m = m; t.mt = mt; t.np = np; t.mp = mp;
        const int K[3] = {np + 16 + mp, np + 16, mp}, N[3] = {np, mp, np};
        t.ok = mp <= 256 && np <= 256 && 2 * mp + np <= 512;
        t.merged = 3 * mp + 2 * np <= 512 && 2 * mp <= 256;
        size_t total = 0;
        for (int p = 0; p < 3; ++p) {
            t.ncols[p] = N[p]; t.ksteps[p] = K[p] / 8; t.nchunks[p] = (K[p] + 31) / 32;
            t.pair_bytes[p] = N[p] * 128 * 2;
            t.off[p] = (int)total;
            total += (size_t)t.nchunks[p] * t.pair_bytes[p];
        }
        const int a_stage = 128 * 128 * 2;
        // tables, per-slot state and barriers behind the rings (tc_carve in qp_admm_tc.cu): 4 mp + 16 np floats, 6 mp doubles,
        // 5 x 128 doubles, 8 x 128 words, 16 barriers
        const int tables = (4 * mp + 16 * np + 48 * mp + 40 * 128 + 32 * 128 + 8 * 16 + 8 + 8 * 16 + 64 + 1023) / 1024 * 1024;
        const int budget = 227 * 1024 - 1024;                      // the dynamic area is re-aligned to 1024 bytes in the kernel
        t.resident_bytes = t.nchunks[0] * t.pair_bytes[0] + t.nchunks[1] * t.pair_bytes[1];
        t.nb_stages = 2;
        if (2 * a_stage + t.resident_bytes + t.pair_bytes[2] + tables <= budget) {
            // small problems: the matrices of products 0 and 1 stay in shared memory; the certificate product (once per
            // round) streams through one or two stages
            t.resident = 1;
            t.b_stage_bytes = t.pair_bytes[2];
            t.nb_stages = 2 * a_stage + t.resident_bytes + 2 * t.pair_bytes[2] + tables <= budget ? 2 : 1;
            t.na_stages = 3 * a_stage + t.resident_bytes + t.nb_stages * t.pair_bytes[2] + tables <= budget ? 3 : 2;
            t.smem_bytes = t.na_stages * a_stage + t.resident_bytes + t.nb_stages * t.b_stage_bytes + tables + 1024;
        } else {
            t.resident = 0;
            t.resident_bytes = 0;
            t.b_stage_bytes = std::max(t.pair_bytes[0], std::max(t.pair_bytes[1], t.pair_bytes[2]));
            t.na_stages = 3 * a_stage + 2 * t.b_stage_bytes + tables <= budget ? 3 : 2;
            t.smem_bytes = t.na_stages * a_stage + 2 * t.b_stage_bytes + tables + 1024;
            if (t.smem_bytes > 227 * 1024) t.ok = 0;
        }
        if (!t.ok) return;
        auto tf32_rn = [](double v) {
            float f = (float)v;
            uint32_t u; memcpy(&u, &f, 4);
            u = (u + 0x1000u) & 0xFFFFE000u;
            memcpy(&f, &u, 4);
            return f;
        };
        auto sw128 = [](int r, int k) { return (r >> 3) * 1024 + (r & 7) * 128 + (((k >> 2) ^ (r & 7)) << 4) + (k & 3) * 4; };
        P.img.assign(total, 0);
        auto put = [&](int p, int r, int k, double v) {
            if (v == 0.0) return;
            unsigned char* base = P.img.data() + t.off[p] + (size_t)(k >> 5) * t.pair_bytes[p];
            const float hi = tf32_rn(v), lo = tf32_rn(v - (double)hi);
            memcpy(base + sw128(r, k & 31), &hi, 4);
            memcpy(base + (size_t)N[p] * 128 + sw128(r, k & 31), &lo, 4);
        };
        // e columns: x0_c as three pieces (3c .. 3c + 2), the constant 1 (12), the disturbance as three pieces (13 .. 15)
        auto put_e = [&](int p, int r, int k0, const double* cx, double c1, double cc) {
            for (int c = 0; c < 4; ++c)
                for (int piece = 0; piece < 3; ++piece) put(p, r, k0 + 3 * c + piece, cx[c]);
            put(p, r, k0 + 12, c1);
            for (int piece = 0; piece < 3; ++piece) put(p, r, k0 + 13 + piece, cc);
        };
        std::vector<double> his(mp, 0.0), gxs((size_t)mp * 4, 0.0), gcs(mp, 0.0);
        P.nwd.assign(mp, -INFINITY); P.einv_g.assign(mp, 0.f); P.row_id.assign(mp, -1);
        for (int r = 0; r < nr; ++r) {
            const int i = prows[r];
            his[r] = Eg[i] * q.hi[i];
            for (int c = 0; c < 4; ++c) gxs[(size_t)r * 4 + c] = Eg[i] * q.Gx[(size_t)i * 4 + c];
            gcs[r] = Eg[i] * q.Gc[i];
            P.nwd[r] = isinf(q.lo[i]) ? -INFINITY : -(float)(Eg[i] * (q.hi[i] - q.lo[i]));
            P.einv_g[r] = (float)(1.0 / Eg[i]);
            P.row_id[r] = i;
        }
        P.his = his; P.gxs = gxs; P.gcs = gcs;
        P.hisf.assign(his.begin(), his.end()); P.gxsf.assign(gxs.begin(), gxs.end()); P.gcsf.assign(gcs.begin(), gcs.end());
        P.lam.assign(np, 0.f); P.lb.assign(np, -INFINITY); P.ub.assign(np, INFINITY);
        P.einv_b.assign(np, 0.f); P.nrl.assign(np, 0.f); P.kfv.assign((size_t)np * 4, 0.0);
        P.var_id.assign(np, -1);
        for (int a = 0; a < nv; ++a) {
            const int j = vars[a];
            P.var_id[a] = j;
            P.lam[a] = (float)lam[j];
            P.lb[a] = isinf(lb_in[j]) ? -INFINITY : (float)(Eb[j] * lb_in[j]);
            P.ub[a] = isinf(ub_in[j]) ? INFINITY : (float)(Eb[j] * ub_in[j]);
            P.einv_b[a] = (float)(1.0 / Eb[j]);
            P.nrl[a] = lam[j] > 0 ? (float)(-1.0 / lam[j]) : 0.f;
            for (int c = 0; c < 4; ++c) {
                double sum = 0;
                for (int k = 0; k < n; ++k) sum += q.Kinv[(size_t)j * n + k] * cs * D[k] * q.F[(size_t)k * 4 + c];
                P.kfv[(size_t)a * 4 + c] = -sum;
            }
        }
        // product 0: x~ = rho K^-1 [diag(lam) V_b + Gs' (V^_g + h)] + kfv x0 (- kfv xref, added by the kernel)
        for (int a = 0; a < nv; ++a) {
            const int ja = vars[a];
            double cx[4] = {P.kfv[(size_t)a * 4], P.kfv[(size_t)a * 4 + 1], P.kfv[(size_t)a * 4 + 2], P.kfv[(size_t)a * 4 + 3]};
            double c1 = 0, cc = 0;
            for (int b2 = 0; b2 < nv; ++b2) {
                const int j = vars[b2];
                if (comp[j] == comp[ja]) put(0, a, b2, rho * q.Kinv[(size_t)ja * n + j] * lam[j]);
            }
            for (int r = 0; r < nr; ++r) {
                const int i = prows[r];
                if (row_vars[i].empty() || row_comp[i] != comp[ja]) continue;
                const double pg = rho * KG[(size_t)ja * m + i];
                put(0, a, np + 16 + r, pg);
                for (int c = 0; c < 4; ++c) cx[c] -= pg * gxs[(size_t)r * 4 + c];
                c1 += pg * his[r];
                cc -= pg * gcs[r];
            }
            put_e(0, a, np, cx, c1, cc);
        }
        // product 1: z^ = Gs x~ - h ;  product 2: Gs' dy
        for (int r = 0; r < nr; ++r) {
            const int i = prows[r];
            for (int a = 0; a < nv; ++a) {
                put(1, r, a, q.Gs64[(size_t)i * n + vars[a]]);
                put(2, a, r, q.Gs64[(size_t)i * n + vars[a]]);
            }
            put_e(1, r, np, &gxs[(size_t)r * 4], -his[r], gcs[r]);
        }
    };
    {
        q.tc_parts.clear();
        std::vector<int> all_vars(n);
        std::iota(all_vars.begin(), all_vars.end(), 0);
        q.tc_parts.emplace_back();
        build_part(all_vars, rows, q.tc_parts[0]);
        if (!q.tc_parts[0].t.ok && ncomp >= 2) {
            std::vector<TcPart> parts(ncomp);
            bool all_ok = true;
            for (int c = 0; c < ncomp && all_ok; ++c) {
                std::vector<int> cv, cr;
                for (int j = 0; j < n; ++j) if (comp[j] == c) cv.push_back(j);
                for (int i : rows) if ((row_vars[i].empty() ? 0 : row_comp[i]) == c) cr.push_back(i);
                build_part(cv, cr, parts[c]);
                all_ok = parts[c].t.ok != 0;
            }
            if (all_ok) q.tc_parts.swap(parts);
        }
        q.tc = q.tc_parts[0].t;
    }

    q.mats_in_smem = GA < 4 && admm_smem_bytes(q, S, true) <= (size_t)226 * 1024;
    q.smem_bytes = admm_smem_bytes(q, S, q.mats_in_smem);
    if (q.smem_bytes > (size_t)227 * 1024) { set_error("carmpc_qp_create: shared-memory budget exceeded"); return CARMPC_ERR_UNSUPPORTED; }
    return CARMPC_OK;
}

}  // namespace carmpc
