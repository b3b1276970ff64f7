// plan.cu — host-side plan of a problem (plan.h).  Host code only: dbat_create uploads what it builds.
#include <algorithm>
#include <cstring>
#include <iterator>
#include <map>

#include "plan.h"

static int fail(std::string& err, int code, const char* msg) {
    err = msg;
    return code;
}

int plan_columns(const dbat_problem_desc* d, ProblemPlan& p, std::string& err) {
    const int nImg = (int)d->nImg, nOP = (int)d->nOP, nObs = (int)d->nIP;
    const int nK = d->nK, nP = d->nP, NC = 5 + nK + nP;
    const bool legacy = (d->distModel == 1 || d->distModel == -1);
    if (!legacy && (d->distModel < 2 || d->distModel > 5))
        return fail(err, DBAT_E_BADARG, "distModel must be -1, 1, 2, 3, 4 or 5");
    if (nK > DBAT_KMAX || nP > DBAT_PMAX || nK < 0 || nP < 0 || nP == 1)
        return fail(err, DBAT_E_UNSUPPORTED, "nK/nP outside the compiled limits");
    if (d->n <= 0 || nImg <= 0) return fail(err, DBAT_E_BADARG, "empty problem");
    p.nImg = nImg; p.nOP = nOP; p.nObs = nObs; p.n = (int)d->n; p.NC = NC; p.legacy = legacy;

    // ---- column maps from the deserialisation indices (multi_res.m:58-63)
    std::vector<int> colIO((size_t)NC * nImg, -1), colEO((size_t)6 * nImg, -1), colOP((size_t)3 * nOP, -1);
    auto fill = [&](std::vector<int>& col, const int64_t* src, const int64_t* dst, int64_t cnt) -> bool {
        for (int64_t k = 0; k < cnt; ++k) {
            const int64_t dd = dst[k] - 1, ss = src[k] - 1;
            if (dd < 0 || dd >= (int64_t)col.size() || ss < 0 || ss >= d->n) return false;
            col[dd] = (int)ss;
        }
        return true;
    };
    if (!fill(colIO, d->IOdes_src, d->IOdes_dest, d->nIOdes) || !fill(colEO, d->EOdes_src, d->EOdes_dest, d->nEOdes) ||
        !fill(colOP, d->OPdes_src, d->OPdes_dest, d->nOPdes))
        return fail(err, DBAT_E_BADARG, "deserialisation index out of range");
    // camera-side unknowns x[0:nC]: everything up to the last IO/EO column (a point-sharded problem
    // lists only its own OP columns, so n - nOPdes would be wrong there)
    int nC = 0;
    for (int c : colIO) nC = std::max(nC, c + 1);
    for (int c : colEO) nC = std::max(nC, c + 1);
    for (int c : colOP) if (c >= 0 && c < nC) return fail(err, DBAT_E_UNSUPPORTED, "x must be ordered [IO;EO;OP]");
    for (int c : colIO) if (c >= nC) return fail(err, DBAT_E_UNSUPPORTED, "x must be ordered [IO;EO;OP]");
    for (int c : colEO) if (c >= nC) return fail(err, DBAT_E_UNSUPPORTED, "x must be ordered [IO;EO;OP]");
    p.nC = nC;

    // ---- observations: 0-based, verify (image, OP) ordering
    p.img_cm.resize(nObs); p.pt_cm.resize(nObs);
    std::vector<char> imgHasObs(nImg, 0);
    for (int k = 0; k < nObs; ++k) {
        const int64_t i = d->IPimg[k] - 1, j = d->IPop[k] - 1;
        if (i < 0 || i >= nImg || j < 0 || j >= nOP) return fail(err, DBAT_E_BADARG, "IPimg/IPop out of range");
        if (k > 0 && (i < p.img_cm[k - 1] || (i == p.img_cm[k - 1] && j <= p.pt_cm[k - 1])))
            return fail(err, DBAT_E_BADARG, "image points must be sorted by (image, OP) without duplicates");
        p.img_cm[k] = (int)i; p.pt_cm[k] = (int)j; imgHasObs[i] = 1;
    }
    // ---- structure checks: one shared IO block; every EO column owned by one image
    p.sh_col.assign(DBAT_NSLOT, -1);
    auto slot_of = [&](int row) { return row < 5 ? row : (row < 5 + nK ? DBAT_SLOT_K + (row - 5) : DBAT_SLOT_P + (row - 5 - nK)); };
    int firstImg = -1;
    for (int i = 0; i < nImg; ++i) if (imgHasObs[i]) { firstImg = i; break; }
    if (legacy) {
        // brown_euler_cam4.m:39-41,186-188: est.IO(:,2:end)=false, EO.cam(:)=1, IP.cam(:)=1
        for (int i = 1; i < nImg; ++i)
            for (int r = 0; r < NC; ++r) colIO[(size_t)i * NC + r] = colIO[r];
        colIO[3] = -1; colIO[4] = -1;          // aspect / skew do not exist in the legacy models
        for (int i = 1; i < nImg; ++i) { colIO[(size_t)i * NC + 3] = -1; colIO[(size_t)i * NC + 4] = -1; }
    }
    // IO column of every (image, slot); one block shared by all images -> fast path, anything else (image-variant
    // parameters, several cameras: IO.struct.block, multi_res.m:92-111) -> general path
    p.io_colx.assign((size_t)nImg * DBAT_NSLOT, -1);
    for (int i = 0; i < nImg; ++i)
        for (int r = 0; r < NC; ++r) p.io_colx[(size_t)i * DBAT_NSLOT + slot_of(r)] = colIO[(size_t)i * NC + r];
    bool general = false;
    for (int r = 0; r < NC; ++r) {
        int v = firstImg >= 0 ? colIO[(size_t)firstImg * NC + r] : -1;
        for (int i = 0; i < nImg; ++i)
            if (imgHasObs[i] && colIO[(size_t)i * NC + r] != v) general = true;
        p.sh_col[slot_of(r)] = v;
    }
    if (general && legacy) return fail(err, DBAT_E_UNSUPPORTED, "the legacy models take one camera");
    if (general) p.sh_col.assign(DBAT_NSLOT, -1);      // no column is "the" shared column of a slot
    p.general = general;
    {
        std::vector<int> owner(nC, -1);
        for (int i = 0; i < nImg; ++i)
            for (int a = 0; a < 6; ++a) {
                const int c = colEO[(size_t)i * 6 + a];
                if (c < 0) continue;
                if (owner[c] >= 0 && owner[c] != i) return fail(err, DBAT_E_UNSUPPORTED, "shared EO blocks are not built yet");
                owner[c] = i;
            }
        int prev = -1;   // EO columns must ascend with (image, element): serialisation order
        for (int i = 0; i < nImg; ++i)
            for (int a = 0; a < 6; ++a) {
                const int c = colEO[(size_t)i * 6 + a];
                if (c < 0) continue;
                if (c <= prev) return fail(err, DBAT_E_UNSUPPORTED, "EO columns must be in serialisation order");
                prev = c;
            }
        if (prev >= 0) {
            int minEO = nC;
            for (int c : colEO) if (c >= 0) minEO = std::min(minEO, c);
            for (int c : p.io_colx) if (c > minEO) return fail(err, DBAT_E_UNSUPPORTED, "IO columns must precede EO columns in x");
        }
    }
    p.io_col = std::move(colIO); p.eo_col = std::move(colEO); p.op_col = std::move(colOP);
    return DBAT_OK;
}

void plan_observations(const dbat_problem_desc* d, ProblemPlan& p, PlanUpload& u) {
    const int nImg = p.nImg, nOP = p.nOP, nObs = p.nObs, NC = p.NC;
    const bool legacy = p.legacy;
    // ---- unique IO records (by value of the whole IO column + pixel size)
    u.ioOfImg.assign(nImg, 0);
    {
        std::map<std::vector<double>, int> seen;
        for (int i = 0; i < nImg; ++i) {
            const int src = legacy ? 0 : i;
            std::vector<double> key(d->IOval + (size_t)src * NC, d->IOval + (size_t)(src + 1) * NC);
            if (p.general) key.push_back((double)i);        // estimated per-image parameters diverge: one record per image
            auto it = seen.find(key);
            if (it == seen.end()) { it = seen.emplace(key, (int)u.rep.size()).first; u.rep.push_back(i); }
            u.ioOfImg[i] = it->second;
        }
    }
    p.nIOrec = (int)u.rep.size();
    u.recs.resize(nImg);
    for (int i = 0; i < nImg; ++i) {
        ImgRec& r = u.recs[i];
        memset(&r, 0, sizeof(ImgRec));
        r.sz = d->pxSize[2 * (size_t)(legacy ? 0 : i)];   // multi_res.m:138 passes sz(1)
        r.szy = legacy ? d->pxSize[1] : r.sz;             // legacy: multiscalepts uses both axes
        r.io = u.ioOfImg[i];
    }

    // ---- weights, orderings, chunks
    u.uv_cm.resize(nObs); u.isig_cm.resize(nObs); u.uv_pm.resize(nObs); u.isig_pm.resize(nObs);
    for (int k = 0; k < nObs; ++k) {
        const int i = p.img_cm[k];
        u.uv_cm[k] = make_double2(d->IPval[2 * (size_t)k], d->IPval[2 * (size_t)k + 1]);
        const int ic = legacy ? 0 : i;
        const double sx = d->IPstd[2 * (size_t)k] * d->pxSize[2 * (size_t)ic];
        const double sy = d->IPstd[2 * (size_t)k + 1] * d->pxSize[2 * (size_t)ic + 1];
        u.isig_cm[k] = make_double2(1.0 / sx, 1.0 / sy);           // buildweightmatrix.m:13-23, R = chol(W)
    }
    p.img_start.assign(nImg + 1, 0);
    for (int k = 0; k < nObs; ++k) p.img_start[p.img_cm[k] + 1]++;
    for (int i = 0; i < nImg; ++i) p.img_start[i + 1] += p.img_start[i];
    p.pt_start.assign(nOP + 1, 0);
    for (int k = 0; k < nObs; ++k) p.pt_start[p.pt_cm[k] + 1]++;
    for (int j = 0; j < nOP; ++j) p.pt_start[j + 1] += p.pt_start[j];
    p.pm2cm.resize(nObs);
    u.img_pm.resize(nObs);
    {
        std::vector<int> fillp(p.pt_start.begin(), p.pt_start.end() - 1);
        for (int k = 0; k < nObs; ++k) {                       // stable: images ascend inside a point
            const int o = fillp[p.pt_cm[k]]++;
            p.pm2cm[o] = k; u.img_pm[o] = p.img_cm[k]; u.uv_pm[o] = u.uv_cm[k]; u.isig_pm[o] = u.isig_cm[k];
        }
    }
    u.img_chunk_start.assign(nImg + 1, 0);
    for (int i = 0; i < nImg; ++i) {
        u.img_chunk_start[i] = (int)u.chunks.size();
        for (int s = p.img_start[i]; s < p.img_start[i + 1]; s += DBAT_CHUNK)
            u.chunks.push_back({i, s, std::min(DBAT_CHUNK, p.img_start[i + 1] - s), 0});
    }
    u.img_chunk_start[nImg] = (int)u.chunks.size();
    // point of every point-major observation
    u.pt_pm.resize(nObs);
    for (int o = 0; o < nObs; ++o) u.pt_pm[o] = p.pt_cm[p.pm2cm[o]];
}

int plan_priors(const dbat_problem_desc* d, ProblemPlan& p, PlanUpload& u, std::string& err) {
    const int nPrior = (int)(d->nPriorIO + d->nPriorEO + d->nPriorOP);
    p.prior_col.resize(nPrior); p.prior_isig.resize(nPrior);
    u.prior_val.resize(nPrior);
    for (int k = 0; k < nPrior; ++k) {
        const int64_t c = d->prior_x[k] - 1;
        if (c < 0 || c >= d->n) return fail(err, DBAT_E_BADARG, "prior_x out of range");
        if (!(d->prior_std[k] > 0)) return fail(err, DBAT_E_BADARG, "prior std must be positive");
        p.prior_col[k] = (int)c; u.prior_val[k] = d->prior_val[k]; p.prior_isig[k] = 1.0 / d->prior_std[k];
    }
    p.m = 2 * p.nObs + nPrior;
    u.col2pt.assign(std::max(1, p.n - p.nC), -1);
    for (int e = 0; e < 3 * p.nOP; ++e) if (p.op_col[e] >= 0) u.col2pt[p.op_col[e] - p.nC] = e;
    return DBAT_OK;
}

int plan_cameras(const dbat_problem_desc* d, ProblemPlan& p, const PlanUpload& u, std::string& err) {
    const int nImg = p.nImg, nC = p.nC;
    // ---- reduced system: co-visibility graph of the images
    covis_graph(nImg, p.nOP, p.pt_start.data(), u.img_pm.data(), p.adjPtr, p.adj);
    std::vector<int64_t>& adjPtr = p.adjPtr; std::vector<int32_t>& adj = p.adj;
    if (d->nCovis > 0 && d->covis_a && d->covis_b) {      // the whole project's graph (sharded problems)
        std::vector<std::vector<int32_t>> nb(nImg);
        for (int i = 0; i < nImg; ++i) nb[i].assign(adj.begin() + adjPtr[i], adj.begin() + adjPtr[i + 1]);
        for (int64_t e = 0; e < d->nCovis; ++e) {
            const int64_t a = d->covis_a[e] - 1, b = d->covis_b[e] - 1;
            if (a < 0 || a >= nImg || b < 0 || b >= nImg) return fail(err, DBAT_E_BADARG, "covis edge out of range");
            if (a == b) continue;
            nb[a].push_back((int32_t)b); nb[b].push_back((int32_t)a);
        }
        adj.clear();
        for (int i = 0; i < nImg; ++i) {
            std::sort(nb[i].begin(), nb[i].end());
            nb[i].erase(std::unique(nb[i].begin(), nb[i].end()), nb[i].end());
            adjPtr[i] = (int64_t)adj.size();
            adj.insert(adj.end(), nb[i].begin(), nb[i].end());
        }
        adjPtr[nImg] = (int64_t)adj.size();
    }
    p.xyz.resize((size_t)3 * nImg);
    for (int i = 0; i < nImg; ++i) for (int a = 0; a < 3; ++a) p.xyz[3 * (size_t)i + a] = d->EOval[6 * (size_t)i + a];
    p.nEO.assign(nImg, 0);
    for (int i = 0; i < nImg; ++i) for (int a = 0; a < 6; ++a) if (p.eo_col[(size_t)i * 6 + a] >= 0) p.nEO[i]++;
    // IO columns: used by one image -> they travel with that image (like its EO elements); used by several ->
    // "global", last in S.  (One shared block: every estimated IO column is global.)
    std::vector<int> users(std::max(1, nC), 0), lastUser(std::max(1, nC), -1);
    for (int i = 0; i < nImg; ++i)
        for (int sl = 0; sl < DBAT_NSLOT; ++sl) {
            const int c = p.io_colx[(size_t)i * DBAT_NSLOT + sl];
            if (c >= 0 && lastUser[c] != i) { users[c]++; lastUser[c] = i; }
        }
    p.glob_x.clear();
    p.colLocalImg.assign(std::max(1, nC), -1);
    for (int c = 0; c < nC; ++c) {
        if (users[c] >= 2 || (users[c] == 1 && !p.general)) p.glob_x.push_back(c);
        else if (users[c] == 1) { p.colLocalImg[c] = lastUser[c]; p.nEO[lastUser[c]]++; }
    }
    return DBAT_OK;
}

ReducedMaps plan_reduced_maps(ProblemPlan& p, const TileSym& sym) {
    const int nImg = p.nImg, nC = p.nC;
    ReducedMaps r;
    r.sh_s.assign(DBAT_NSLOT, -1); r.eo_s.assign((size_t)6 * nImg, -1); r.s2x.assign(sym.ld, -1);
    r.cam_colx.assign((size_t)DBAT_NCAM * nImg, -1); r.cam_s.assign((size_t)DBAT_NCAM * nImg, -1);
    std::vector<int>& x2s = p.x2s;
    x2s.assign(std::max(1, nC), -1);
    for (size_t k = 0; k < p.glob_x.size(); ++k) x2s[p.glob_x[k]] = sym.ioS + (int)k;     // global IO columns, x order
    for (int i = 0; i < nImg; ++i) {
        int q = 0;
        for (int a = 0; a < 6; ++a) {
            const int c = p.eo_col[(size_t)i * 6 + a];
            if (c >= 0) { r.eo_s[(size_t)i * 6 + a] = sym.imgS[i] + q; x2s[c] = sym.imgS[i] + q; ++q; }
        }
        for (int sl = 0; sl < DBAT_NSLOT; ++sl) {             // this image's own IO columns follow its EO elements
            const int c = p.io_colx[(size_t)i * DBAT_NSLOT + sl];
            if (c >= 0 && p.colLocalImg[c] == i && x2s[c] < 0) { x2s[c] = sym.imgS[i] + q; ++q; }
        }
    }
    for (int c = 0; c < nC; ++c) if (x2s[c] >= 0) r.s2x[x2s[c]] = c;
    for (int sl = 0; sl < DBAT_NSLOT; ++sl) if (p.sh_col[sl] >= 0) r.sh_s[sl] = x2s[p.sh_col[sl]];
    for (int i = 0; i < nImg; ++i)
        for (int a = 0; a < DBAT_NCAM; ++a) {
            const int c = a < DBAT_NSLOT ? p.io_colx[(size_t)i * DBAT_NSLOT + a] : p.eo_col[(size_t)i * 6 + a - DBAT_NSLOT];
            r.cam_colx[(size_t)i * DBAT_NCAM + a] = c;
            r.cam_s[(size_t)i * DBAT_NCAM + a] = c >= 0 ? x2s[c] : -1;
        }
    return r;
}

void plan_point_blocks(const ProblemPlan& p, PlanUpload& u) {
    // point-side assembly blocks: runs [begin, end) of whole points with at most DBAT_PSB observations (and at most
    // DBAT_PSB / 2 points); a point with more observations than that goes to the one-thread-per-point kernel
    std::vector<int>& pairs = u.psb_pt; std::vector<int>& bigp = u.psbig;
    int begin = 0, cnt = 0;
    auto close = [&](int end) { if (end > begin) { pairs.push_back(begin); pairs.push_back(end); } begin = end; cnt = 0; };
    for (int j = 0; j < p.nOP; ++j) {
        const int k = p.pt_start[j + 1] - p.pt_start[j];
        if (k > DBAT_PSB) { close(j); bigp.push_back(j); begin = j + 1; continue; }
        if (cnt + k > DBAT_PSB || j - begin >= DBAT_PSB / 2) close(j);
        cnt += k;
    }
    close(p.nOP);
    u.nPsb = (int)pairs.size() / 2;
    u.nPsbig = (int)bigp.size();
    if (pairs.empty()) pairs.assign(2, 0);
    if (bigp.empty()) bigp.push_back(0);
}

void plan_schur_windows(ProblemPlan& p, PlanUpload& u, const TileSym& sym, const PlanOpts& opts) {
    const int nImg = p.nImg, nOP = p.nOP, nObs = p.nObs;
    const std::vector<int>& imgRank = sym.imgRank;
    const std::vector<int>& img_pm = u.img_pm;
    // grouped Schur index: estimated points sorted by (ray count, image list)
    std::vector<int>& cand = u.grp_pt; std::vector<int>& big = u.big_pt;
    cand.reserve(nOP);
    const int maxm = opts.grpMaxM;
    for (int j = 0; j < nOP; ++j) {
        const int k = p.pt_start[j + 1] - p.pt_start[j];
        const int* oc = &p.op_col[3 * (size_t)j];
        if (k == 0 || (oc[0] < 0 && oc[1] < 0 && oc[2] < 0)) continue;
        (k <= maxm ? cand : big).push_back(j);
    }
    const int* ps = p.pt_start.data();
    // image lists in elimination-order rank (ascending inside a point): the union of a group is then
    // ascending in S order, which the lower-triangular window blocks of k_schur_win rely on
    std::vector<int> rk(std::max(1, nObs));
    for (int j = 0; j < nOP; ++j) {
        for (int o = ps[j]; o < ps[j + 1]; ++o) rk[o] = imgRank[img_pm[o]];
        std::sort(rk.begin() + ps[j], rk.begin() + ps[j + 1]);
    }
    const int* im = rk.data();
    // lexicographic order of the (ascending) image lists: points with similar lists become neighbours
    std::sort(cand.begin(), cand.end(), [&](int a, int b) {
        const int ka = ps[a + 1] - ps[a], kb = ps[b + 1] - ps[b];
        const int* la = im + ps[a]; const int* lb = im + ps[b];
        for (int t = 0; t < std::min(ka, kb); ++t) if (la[t] != lb[t]) return la[t] < lb[t];
        return ka != kb ? ka < kb : a < b;
    });
    // greedy groups of consecutive points: at most gcap points, union of their image lists at most
    // `mu` images (a single point always fits).  A point that lacks an image of the union simply
    // has zero rows there.
    const int gcap = std::max(1, std::min(WIN_GP, (int)(cand.size() / (148 * 8))));
    const int mu = 12;
    std::vector<int> gstart, gimg_off, gimg, uni, tmp;
    std::vector<unsigned char> slot(std::max(1, nObs), 0);
    gstart.push_back(0); gimg_off.push_back(0);
    auto close_group = [&](size_t end) {
        for (size_t i = gstart.back(); i < end; ++i) {
            const int j = cand[i];
            for (int o = ps[j]; o < ps[j + 1]; ++o)
                slot[o] = (unsigned char)(std::lower_bound(uni.begin(), uni.end(), imgRank[img_pm[o]]) - uni.begin());
        }
        for (int r : uni) gimg.push_back(sym.imgOrder[r]);
        gimg_off.push_back((int)gimg.size());
        p.grpMaxPts = std::max(p.grpMaxPts, (int)end - gstart.back());
        gstart.push_back((int)end);
        u.grpMaxRays = std::max(u.grpMaxRays, (int)uni.size());
    };
    for (size_t i = 0; i < cand.size(); ++i) {
        const int j = cand[i];
        tmp.clear();
        std::set_union(uni.begin(), uni.end(), im + ps[j], im + ps[j + 1], std::back_inserter(tmp));
        const int cnt = (int)(i - gstart.back());
        if (cnt > 0 && ((int)tmp.size() > mu || cnt >= gcap)) {
            close_group(i);
            uni.assign(im + ps[j], im + ps[j + 1]);
        } else {
            uni.swap(tmp);
        }
    }
    if (!cand.empty()) close_group(cand.size());
    const bool noCand = cand.empty();
    if (noCand) { cand.push_back(0); gstart.assign(1, 0); gimg_off.assign(1, 0); gimg.push_back(0); }
    if (big.empty()) big.push_back(0); else u.nBig = (int)big.size();
    const int nGrp = (int)gstart.size() - 1;
    // ---- window Schur (schur_win.cu): group headers, clusters of consecutive groups whose unions span at most
    //      WIN_MAXW images, and the fixed-order reduction index of the cluster images
    u.nCand = noCand ? 0 : (int)cand.size();
    std::vector<WinHdr>& hdr = u.win_hdr;
    hdr.resize((size_t)std::max(1, nGrp));
    std::vector<int>& clu_grp = u.clu_grp; std::vector<int>& clu_img_off = u.clu_img_off; std::vector<int>& clu_img = u.clu_img;
    std::vector<long long>& clu_stg = u.clu_stg;
    clu_grp.assign(1, 0); clu_img_off.assign(1, 0); clu_stg.assign(1, 0);
    struct Contrib { long long key, off; };
    std::vector<Contrib> contrib;
    std::vector<std::pair<int, long long>> icontrib;         // (image, staging offset of its shared rows)
    const std::vector<int>& imgOrder = sym.imgOrder;
    for (int g = 0; g < nGrp; ++g) {
        WinHdr& H = hdr[g];
        memset(&H, 0, sizeof(H));
        memset(H.obsOf, 255, sizeof(H.obsOf));
        H.m = gimg_off[g + 1] - gimg_off[g];
        H.ng = gstart[g + 1] - gstart[g];
        H.p0 = gstart[g];
        for (int gi = 0; gi < H.ng; ++gi) {
            const int j = cand[gstart[g] + gi];
            H.j[gi] = j; H.ob[gi] = ps[j];
            for (int o = ps[j]; o < ps[j + 1]; ++o) H.obsOf[gi][slot[o]] = (unsigned char)(o - ps[j]);
        }
    }
    {
        const int capG = std::max(4, std::min(48, nGrp / (148 * 8)));
        std::vector<int> win, tmpw, rg;
        unsigned char bm[WIN_MAXW][WIN_MAXW];
        auto close_cluster = [&](int gEnd) {
            const int mw = (int)win.size();
            const long long base = clu_stg.back(), nb36 = (long long)(mw * (mw + 1) / 2) * 36;
            memset(bm, 0, sizeof(bm));
            for (int g = clu_grp.back(); g < gEnd; ++g) {
                WinHdr& H = hdr[g];
                for (int k = 0; k < H.m; ++k)
                    H.wslot[k] = (unsigned char)(std::lower_bound(win.begin(), win.end(), imgRank[gimg[gimg_off[g] + k]]) - win.begin());
                for (int gi = 0; gi < H.ng; ++gi) {
                    const int j = H.j[gi];
                    for (int o1 = ps[j]; o1 < ps[j + 1]; ++o1)
                        for (int o2 = ps[j]; o2 < ps[j + 1]; ++o2) {
                            const int wa = H.wslot[slot[o1]], wb = H.wslot[slot[o2]];
                            if (wa >= wb) bm[wa][wb] = 1;
                        }
                }
            }
            for (int wa = 0; wa < mw; ++wa)
                for (int wb = 0; wb <= wa; ++wb)
                    if (bm[wa][wb]) contrib.push_back({(long long)win[wa] * nImg + win[wb], base + (long long)(wa * (wa + 1) / 2 + wb) * 36});
            for (int w = 0; w < mw; ++w) {
                clu_img.push_back(imgOrder[win[w]]);
                icontrib.push_back({imgOrder[win[w]], base + nb36 + 6 * w});
            }
            clu_img_off.push_back((int)clu_img.size());
            clu_stg.push_back(base + nb36 + 16 * 6 * WIN_MAXW + 256);
            clu_grp.push_back(gEnd);
        };
        for (int g = 0; g < nGrp; ++g) {
            rg.clear();
            for (int k = gimg_off[g]; k < gimg_off[g + 1]; ++k) rg.push_back(imgRank[gimg[k]]);
            tmpw.clear();
            std::set_union(win.begin(), win.end(), rg.begin(), rg.end(), std::back_inserter(tmpw));
            const int cnt = g - clu_grp.back();
            if (cnt > 0 && ((int)tmpw.size() > WIN_MAXW || cnt >= capG)) { close_cluster(g); win = rg; }
            else win.swap(tmpw);
        }
        if (nGrp > 0) close_cluster(nGrp);
    }
    u.nClu = (int)clu_grp.size() - 1;
    std::stable_sort(contrib.begin(), contrib.end(), [](const Contrib& a, const Contrib& b) { return a.key < b.key; });
    u.red_off.assign(std::max<size_t>(1, contrib.size()), 0);
    for (size_t k = 0; k < contrib.size(); ++k) {
        if (k == 0 || contrib[k].key != contrib[k - 1].key) {
            u.red_ptr.push_back((int)k);
            u.red_imgA.push_back(imgOrder[(int)(contrib[k].key / nImg)]);
            u.red_imgB.push_back(imgOrder[(int)(contrib[k].key % nImg)]);
        }
        u.red_off[k] = contrib[k].off;
    }
    u.nRedBlk = (int)u.red_ptr.size();
    u.red_ptr.push_back((int)contrib.size());
    if (u.red_imgA.empty()) { u.red_imgA.push_back(0); u.red_imgB.push_back(0); }
    std::stable_sort(icontrib.begin(), icontrib.end(), [](const std::pair<int, long long>& a, const std::pair<int, long long>& b) { return a.first < b.first; });
    u.redi_ptr.assign(nImg + 1, 0);
    u.redi_off.assign(std::max<size_t>(1, icontrib.size()), 0);
    for (size_t k = 0; k < icontrib.size(); ++k) { u.redi_ptr[icontrib[k].first + 1]++; u.redi_off[k] = icontrib[k].second; }
    for (int i = 0; i < nImg; ++i) u.redi_ptr[i + 1] += u.redi_ptr[i];
    if (clu_img.empty()) clu_img.push_back(0);
    // launch order of the clusters: most groups first
    u.clu_order.assign((size_t)std::max(1, u.nClu), 0);
    for (int c = 0; c < u.nClu; ++c) u.clu_order[c] = c;
    std::stable_sort(u.clu_order.begin(), u.clu_order.begin() + u.nClu, [&](int a, int b) { return clu_grp[a + 1] - clu_grp[a] > clu_grp[b + 1] - clu_grp[b]; });
}

bool plan_same_order(const ProblemPlan& p, const TileSym& a, const TileSym& b) {
    std::vector<int> oa, ob;
    for (int i : a.imgOrder) if (p.nEO[i] > 0) oa.push_back(i);
    for (int i : b.imgOrder) if (p.nEO[i] > 0) ob.push_back(i);
    return oa == ob;
}

bool plan_eval_compact(const ProblemPlan& p, int nK, int nP, const PlanOpts& opts) {
    // one shared IO block whose estimated slots all lie in f, pp, b1, K1-K3, P1-P2
    bool ok = !p.general && nK <= 3 && nP <= 2 && !opts.evalGeneric;
    for (int sl = 0; sl < DBAT_NSLOT; ++sl) if (p.sh_col[sl] >= 0 && !((0x0CEFu >> sl) & 1)) ok = false;
    return ok;
}

int plan_partials(const ProblemPlan& p, const PlanUpload& u) {
    return std::max(2 * ((std::max(p.nObs, p.n) + 255) / 256),
                    2 * (u.nPsb + (u.nPsbig + 127) / 128 + (p.nOP + 127) / 128 + 1) + 2 * ((p.nImg + 3) / 4 + 1)) + 64;
}
