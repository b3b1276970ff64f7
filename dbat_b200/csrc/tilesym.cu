// tilesym.cu — host-only: ordering + symbolic tile factorisation of the reduced camera system
// (see tilesym.h).  Runs once per problem at dbat_create.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <vector>

#include "../../include/dbat_gpu.h"
#include "tilesym.h"

void covis_graph(int nImg, int nOP, const int* pt_start, const int* img_pm, std::vector<int64_t>& adjPtr,
                 std::vector<int32_t>& adj) {
    std::vector<uint64_t> edges;
    for (int j = 0; j < nOP; ++j) {
        const int a0 = pt_start[j], a1 = pt_start[j + 1];
        for (int a = a0; a < a1; ++a)
            for (int b = a + 1; b < a1; ++b) {
                const uint32_t x = (uint32_t)img_pm[a], y = (uint32_t)img_pm[b];
                if (x != y) edges.push_back(((uint64_t)std::min(x, y) << 32) | std::max(x, y));
            }
        if (edges.size() > ((size_t)1 << 24)) {            // keep the working set bounded
            std::sort(edges.begin(), edges.end());
            edges.erase(std::unique(edges.begin(), edges.end()), edges.end());
        }
    }
    std::sort(edges.begin(), edges.end());
    edges.erase(std::unique(edges.begin(), edges.end()), edges.end());
    adjPtr.assign((size_t)nImg + 1, 0);
    for (uint64_t e : edges) { ++adjPtr[(size_t)(e >> 32) + 1]; ++adjPtr[(size_t)(e & 0xffffffffu) + 1]; }
    std::partial_sum(adjPtr.begin(), adjPtr.end(), adjPtr.begin());
    adj.assign((size_t)adjPtr[(size_t)nImg], 0);
    std::vector<int64_t> fill(adjPtr.begin(), adjPtr.end() - 1);
    for (uint64_t e : edges) {
        const int32_t x = (int32_t)(e >> 32), y = (int32_t)(e & 0xffffffffu);
        adj[(size_t)fill[(size_t)x]++] = y;
        adj[(size_t)fill[(size_t)y]++] = x;
    }
}

namespace {

struct Graph {
    int n; const int64_t* ptr; const int32_t* adj;
    int64_t deg(int v) const { return ptr[v + 1] - ptr[v]; }
};

// BFS inside the node set marked with `tag` in mark[]; returns the visit order, level[] filled for visited nodes
static void bfs(const Graph& g, const std::vector<int>& mark, int tag, int root, std::vector<int>& level,
                std::vector<int>& order) {
    order.clear();
    order.push_back(root);
    level[root] = 0;
    // visited = level >= 0 within this call: the caller resets level[] of the set to -1 beforehand
    for (size_t head = 0; head < order.size(); ++head) {
        const int v = order[head];
        for (int64_t k = g.ptr[v]; k < g.ptr[v + 1]; ++k) {
            const int u = g.adj[k];
            if (mark[u] == tag && level[u] < 0) { level[u] = level[v] + 1; order.push_back(u); }
        }
    }
}

// George-Liu pseudo-peripheral node of the component of `start`; leaves level[] / order of the final BFS
static int pseudo_peripheral(const Graph& g, const std::vector<int>& mark, int tag, int start,
                             std::vector<int>& level, std::vector<int>& order) {
    int root = start;
    bfs(g, mark, tag, root, level, order);
    int ecc = level[order.back()];
    for (int it = 0; it < 8; ++it) {
        int cand = -1;
        for (size_t k = order.size(); k-- > 0;) {
            const int v = order[k];
            if (level[v] != ecc) break;
            if (cand < 0 || g.deg(v) < g.deg(cand)) cand = v;
        }
        std::vector<int> saved(order);
        for (int v : saved) level[v] = -1;
        bfs(g, mark, tag, cand, level, order);
        const int e2 = level[order.back()];
        if (e2 > ecc) { root = cand; ecc = e2; continue; }
        // keep the BFS from `root`
        for (int v : order) level[v] = -1;
        bfs(g, mark, tag, root, level, order);
        break;
    }
    return root;
}

struct Orderer {
    const Graph& g;
    int leaf;
    std::vector<int> mark, level;
    int nextTag = 1;
    std::vector<std::vector<int>> segs;       // elimination order as a list of segments
    std::vector<int> segOwner;                // owning part of every segment, -1 = above the cut ("top")
    int cutDepth = 0;                         // the tree is cut into 2^cutDepth parts
    Orderer(const Graph& gg, int lf) : g(gg), leaf(lf), mark(gg.n, 0), level(gg.n, -1) {}

    // nodes: a node set (all currently marked with `tag`); nd = dissect, else one RCM segment.
    // depth / path: position in the dissection tree (path = bits of the left/right choices so far)
    void run(std::vector<int> nodes, int tag, bool nd, int depth = 0, int path = 0) {
        const int ownerHere = depth >= cutDepth ? (path >> (depth - cutDepth)) : (path << (cutDepth - depth));
        // split into connected components first
        for (int v : nodes) level[v] = -1;
        std::vector<int> order;
        std::vector<std::vector<int>> comps;
        for (int s : nodes) {
            if (level[s] >= 0) continue;
            bfs(g, mark, tag, s, level, order);
            comps.push_back(order);
        }
        for (auto& comp : comps) {
            const int ctag = nextTag++;
            for (int v : comp) { mark[v] = ctag; level[v] = -1; }
            pseudo_peripheral(g, mark, ctag, comp[0], level, order);
            const int ecc = level[order.back()];
            if (!nd || (int)comp.size() <= leaf || ecc < 2) {
                segs.emplace_back(order.rbegin(), order.rend());      // reverse Cuthill-McKee-like
                segOwner.push_back(ownerHere);
                continue;
            }
            // separator = one BFS level, chosen for balance among the interior levels; only its nodes
            // with a neighbour in the next level have to stay in the separator
            std::vector<int> cnt(ecc + 1, 0);
            for (int v : comp) cnt[level[v]]++;
            std::vector<int64_t> cum(ecc + 2, 0);
            for (int l = 0; l <= ecc; ++l) cum[l + 1] = cum[l] + cnt[l];
            int best = 1; double bestCost = 1e300;
            for (int l = 1; l < ecc; ++l) {
                const double a = (double)cum[l], b = (double)(comp.size() - cum[l + 1]);
                const double imb = std::abs(a - b) / (double)comp.size();
                const double cost = imb + 0.5 * (double)cnt[l] / (double)comp.size();
                if (cost < bestCost) { bestCost = cost; best = l; }
            }
            std::vector<int> A, B, S;
            for (int v : order) {
                if (level[v] < best) A.push_back(v);
                else if (level[v] > best) B.push_back(v);
                else {
                    bool touches = false;
                    for (int64_t k = g.ptr[v]; k < g.ptr[v + 1] && !touches; ++k) {
                        const int u = g.adj[k];
                        if (mark[u] == ctag && level[u] == best + 1) touches = true;
                    }
                    (touches ? S : A).push_back(v);
                }
            }
            if (A.empty() || B.empty()) { segs.emplace_back(order.rbegin(), order.rend()); segOwner.push_back(ownerHere); continue; }
            const int ta = nextTag++, tb = nextTag++;
            for (int v : A) mark[v] = ta;
            for (int v : B) mark[v] = tb;
            for (int v : S) mark[v] = -1;
            run(A, ta, true, depth + 1, 2 * path);
            run(B, tb, true, depth + 1, 2 * path + 1);
            segs.push_back(S);
            segOwner.push_back(depth >= cutDepth ? ownerHere : -1);   // a separator above the cut belongs to everybody
        }
    }
};

}  // namespace

#ifndef TC_CHUNK
#define TC_CHUNK 10                    // terms per partial-sum link of a long task (see emit_chain)
#endif
int tile_symbolic(int nImg, const int64_t* adjPtr, const int32_t* adj, const int* nEO, int nIO, int mode,
                  int leafImages, TileSym& out, int nParts, int myPart) {
    const int T = TC_T;
    out = TileSym();
    int nCamCols = 0;
    for (int i = 0; i < nImg; ++i) nCamCols += nEO[i];
    if (mode < 0) mode = (nCamCols >= 24 * T) ? 2 : 0;      // small systems: one dense front
    // the tree can only be cut where it was dissected; parts = largest power of two <= nParts
    int cutDepth = 0;
    if (mode == 2) while ((2 << cutDepth) <= nParts) ++cutDepth;
    out.nParts = 1 << cutDepth;
    out.myPart = myPart < out.nParts ? myPart : -2;           // a rank beyond the parts owns nothing
    out.order_mode = mode;
    Graph g{nImg, adjPtr, adj};
    // ---- elimination order as segments; every segment starts on a tile boundary when dissecting
    std::vector<std::vector<int>> segs;
    std::vector<int> segOwner;
    if (mode == 0) {
        segs.emplace_back(nImg);
        std::iota(segs[0].begin(), segs[0].end(), 0);
        segOwner.push_back(-1);
    } else {
        Orderer o(g, leafImages);
        o.cutDepth = cutDepth;
        std::vector<int> all(nImg);
        std::iota(all.begin(), all.end(), 0);
        for (int v : all) o.mark[v] = 0;
        o.nextTag = 1;
        o.run(all, 0, mode == 2);
        segs.swap(o.segs);
        segOwner.swap(o.segOwner);
        if (cutDepth == 0) std::fill(segOwner.begin(), segOwner.end(), -1);
    }
    out.nSeg = (int)segs.size();
    out.imgOrder.clear(); out.imgRank.assign(nImg, -1); out.imgS.assign(nImg, -1);
    const bool align = mode == 2 && segs.size() > 1;
    int cur = 0;
    std::vector<int> colOwnerS;                       // owner of every S index handed out so far
    for (size_t q = 0; q < segs.size(); ++q) {
        auto& sg = segs[q];
        int cols = 0;
        for (int v : sg) cols += nEO[v];
        if (cols == 0) { for (int v : sg) { out.imgRank[v] = (int)out.imgOrder.size(); out.imgOrder.push_back(v); } continue; }
        if (align) {
            const int prevOwner = colOwnerS.empty() ? -1 : colOwnerS.back();
            cur = (cur + T - 1) / T * T;
            colOwnerS.resize(cur, prevOwner);         // the alignment padding stays with the segment before it
        }
        for (int v : sg) {
            out.imgRank[v] = (int)out.imgOrder.size();
            out.imgOrder.push_back(v);
            if (nEO[v] > 0) { out.imgS[v] = cur; cur += nEO[v]; }
        }
        colOwnerS.resize(cur, segOwner[q]);
    }
    if ((int)out.imgOrder.size() != nImg) return DBAT_E_BADARG;
    if (cutDepth > 0) {                                   // the IO block and the rhs row never share a tile column with an owned segment
        const int prevOwner = colOwnerS.empty() ? -1 : colOwnerS.back();
        cur = (cur + T - 1) / T * T;
        colOwnerS.resize(cur, prevOwner);
    }
    out.ioS = cur;
    const int nEnd = cur + nIO;                       // unknowns occupy [0, nEnd) minus the alignment padding
    out.nS = nCamCols + nIO;
    out.ld = (nEnd + 1 + T - 1) / T * T;
    out.nT = out.ld / T;
    const int nT = out.nT;
    colOwnerS.resize(out.ld, -1);
    out.colOwner.assign(nT, -1);
    for (int J = 0; J < nT; ++J) {
        int ow = colOwnerS[(size_t)J * T];
        for (int k = 1; k < T; ++k) if (colOwnerS[(size_t)J * T + k] != ow) ow = -1;      // mixed (cannot happen when aligned)
        out.colOwner[J] = ow;
    }
    out.s2kind.assign(out.ld, 0);
    for (int i = 0; i < nImg; ++i) for (int a = 0; a < nEO[i]; ++a) out.s2kind[out.imgS[i] + a] = 1;
    for (int a = 0; a < nIO; ++a) out.s2kind[out.ioS + a] = 1;
    out.s2kind[out.ld - 1] = 2;

    // ---- tile pattern of S (lower triangle incl. diagonal) as bitsets per tile column
    const int W = (nT + 63) / 64;
    std::vector<uint64_t> colS((size_t)nT * W, 0), colL;
    auto setbit = [&](std::vector<uint64_t>& b, int I, int J) { b[(size_t)J * W + (I >> 6)] |= (uint64_t)1 << (I & 63); };
    auto getbit = [&](const std::vector<uint64_t>& b, int I, int J) { return (b[(size_t)J * W + (I >> 6)] >> (I & 63)) & 1; };
    auto mark_pair = [&](int sa, int na, int sb, int nb) {       // S ranges [sa, sa+na) x [sb, sb+nb)
        const int a0 = sa / T, a1 = (sa + na - 1) / T, b0 = sb / T, b1 = (sb + nb - 1) / T;
        for (int I = a0; I <= a1; ++I)
            for (int J = b0; J <= b1; ++J) { if (I >= J) setbit(colS, I, J); else setbit(colS, J, I); }
    };
    for (int i = 0; i < nImg; ++i) {
        if (nEO[i] == 0) continue;
        mark_pair(out.imgS[i], nEO[i], out.imgS[i], nEO[i]);
        for (int64_t k = adjPtr[i]; k < adjPtr[i + 1]; ++k) {
            const int u = adj[k];
            if (u < i && nEO[u] > 0) mark_pair(out.imgS[i], nEO[i], out.imgS[u], nEO[u]);
        }
    }
    for (int J = 0; J < nT; ++J) {
        setbit(colS, J, J);
        setbit(colS, nT - 1, J);                                     // rhs row
        if (nIO > 0) for (int I = out.ioS / T; I <= (out.ioS + nIO - 1) / T; ++I) if (I >= J) setbit(colS, I, J);
    }
    // ---- symbolic factorisation: the parent column inherits the rows below it
    colL = colS;
    std::vector<int> parent(nT, -1);
    for (int J = 0; J < nT; ++J) {
        int p = -1;
        for (int I = J + 1; I < nT && p < 0; ++I) if (getbit(colL, I, J)) p = I;
        parent[J] = p;
        if (p < 0) continue;
        for (int w = p >> 6; w < W; ++w) {
            uint64_t bits = colL[(size_t)J * W + w];
            if (w == (p >> 6)) bits &= ~(((uint64_t)2 << (p & 63)) - 1);     // rows > p only
            colL[(size_t)p * W + w] |= bits;
        }
    }
    out.level.assign(nT, 0);
    for (int J = 0; J < nT; ++J) if (parent[J] >= 0) out.level[parent[J]] = std::max(out.level[parent[J]], out.level[J] + 1);
    out.depth = 0;
    for (int J = 0; J < nT; ++J) out.depth = std::max(out.depth, out.level[J] + 1);
    // an owned column may only have rows in columns of the same owner or in top columns (guaranteed by the
    // dissection; verified here because everything distributed rests on it)
    for (int J = 0; J < nT; ++J) {
        if (out.colOwner[J] < 0) continue;
        for (int I = J + 1; I < nT; ++I)
            if (getbit(colL, I, J) && out.colOwner[I] >= 0 && out.colOwner[I] != out.colOwner[J]) return DBAT_E_STATE;
    }

    // ---- slots: [top S | top fill | owned S by part | owned fill by part]
    out.tix.assign((size_t)nT * nT, -1);
    out.slotI.clear(); out.slotJ.clear();
    out.ownSBegin.assign(out.nParts + 1, 0);
    auto add_tiles = [&](int owner, bool wantS) {
        for (int J = 0; J < nT; ++J) {
            if (out.colOwner[J] != owner) continue;
            for (int I = J; I < nT; ++I) {
                if (!getbit(colL, I, J)) continue;
                if ((getbit(colS, I, J) != 0) != wantS) continue;
                out.tix[(size_t)I * nT + J] = (int)out.slotI.size();
                out.slotI.push_back(I); out.slotJ.push_back(J);
            }
        }
    };
    add_tiles(-1, true);  out.nTopS = (int)out.slotI.size();
    add_tiles(-1, false); out.nTop = (int)out.slotI.size();
    for (int gpart = 0; gpart < out.nParts; ++gpart) { out.ownSBegin[gpart] = (int)out.slotI.size(); add_tiles(gpart, true); }
    out.ownSBegin[out.nParts] = (int)out.slotI.size();
    out.nOwnS = (int)out.slotI.size() - out.nTop;
    for (int gpart = 0; gpart < out.nParts; ++gpart) add_tiles(gpart, false);
    out.nSlots = (int)out.slotI.size();
    out.nSlotsS = out.nTopS + out.nOwnS;
    out.colPtr.assign(nT + 1, 0); out.colSlot.clear();
    std::vector<std::vector<int>> rowCols(nT);                       // per tile row: its columns k < row, ascending
    for (int J = 0; J < nT; ++J) {
        for (int I = J; I < nT; ++I)
            if (getbit(colL, I, J)) { out.colSlot.push_back(out.tix[(size_t)I * nT + J]); if (I > J) rowCols[I].push_back(J); }
        out.colPtr[J + 1] = (int)out.colSlot.size();
    }
    // ... and every column an owned column depends on must belong to the same part (a top column may only sit above)
    for (int J = 0; J < nT; ++J) {
        if (out.colOwner[J] < 0) continue;
        for (int k : rowCols[J]) if (out.colOwner[k] != out.colOwner[J]) return DBAT_E_STATE;
    }
    // ---- task lists: columns by (level, index); within a column the diagonal tile first, then rows ascending.
    //   phase 1: every tile of this part's own columns (all their terms lie in the same subtree), then one
    //            partial-sum task per top tile that has terms in this part's subtree;
    //   phase 2: every tile of the top columns with the terms that lie in top columns (after the partial sums of
    //            all parts have been added up).  One part: everything is top, phase 1 is empty.
    std::vector<int> cols(nT);
    std::iota(cols.begin(), cols.end(), 0);
    std::stable_sort(cols.begin(), cols.end(), [&](int a, int b) { return out.level[a] < out.level[b]; });
    out.taskI.clear(); out.taskJ.clear(); out.taskMode.clear(); out.taskWait.clear(); out.taskSet.clear(); out.taskInit.clear(); out.termPtr.assign(1, 0); out.termA.clear(); out.termB.clear();
    const int me = out.myPart;
    struct Tmp { double key; int I, J, mode, wait, set, init; std::vector<int> a, b, lev; };
    auto inS = [&](int slot) { return slot < out.nTopS || (slot >= out.nTop && slot < out.nTop + out.nOwnS); };
    auto collect = [&](int I, int J, int mode_, int termOwner, Tmp& t) -> bool {   // terms whose column k has owner termOwner
        const std::vector<int>& ri = rowCols[I];
        const std::vector<int>& rj = rowCols[J];
        size_t a = 0, b = 0;
        std::vector<std::pair<int, int>> tk;                       // (level, k) of the common columns
        t.I = I; t.J = J; t.mode = mode_; t.a.clear(); t.b.clear(); t.lev.clear();
        while (a < ri.size() && b < rj.size() && ri[a] < J && rj[b] < J) {
            if (ri[a] < rj[b]) ++a;
            else if (ri[a] > rj[b]) ++b;
            else {
                if (out.colOwner[ri[a]] == termOwner) tk.emplace_back(out.level[ri[a]], ri[a]);
                ++a; ++b;
            }
        }
        // in the order the tiles become available (elimination-tree level), not by index: a task must not sit on a
        // tile of a late subtree while others are ready
        std::stable_sort(tk.begin(), tk.end());
        for (auto& lk : tk) {
            t.a.push_back(out.tix[(size_t)I * nT + lk.second]);
            t.b.push_back(out.tix[(size_t)J * nT + lk.second]);
            t.lev.push_back(lk.first);
        }
        return !(mode_ == 1 && t.a.empty());                       // nothing to add from this subtree: no task
    };
    // A task with many terms becomes a chain: partial sums of <= TC_CHUNK terms each, written back to the tile and
    // released through an auxiliary flag, then the task proper with the last terms.  Every link sorts into the list
    // right after the last column it reads, so the early links run long before the tile's turn and the link on the
    // critical path is short.
    static_assert(TC_CHUNK >= 2, "a partial-sum chain link needs at least two terms");
    int nAux = 0;
    auto emit_chain = [&](const Tmp& t, bool alwaysFromTile, std::vector<Tmp>& list) {
        const int slot = out.tix[(size_t)t.I * nT + t.J];
        const int n = (int)t.a.size();
        const int firstInit = (alwaysFromTile || inS(slot)) ? 1 : 0;
        const double finalKey = t.mode == 0 ? (double)out.level[t.J] : (n ? t.lev.back() + 0.5 : 0.0);
        if (n <= TC_CHUNK + TC_CHUNK / 2) {
            Tmp u = t; u.key = finalKey; u.wait = -1; u.set = -1; u.init = firstInit;
            list.push_back(u);
            return;
        }
        int prev = -1;
        for (int b0 = 0; b0 < n; b0 += TC_CHUNK) {
            int b1 = std::min(n, b0 + TC_CHUNK);
            if (n - b1 < TC_CHUNK / 2) b1 = n;                     // no tiny last link
            Tmp u;
            u.I = t.I; u.J = t.J;
            u.a.assign(t.a.begin() + b0, t.a.begin() + b1);
            u.b.assign(t.b.begin() + b0, t.b.begin() + b1);
            u.wait = prev; u.init = prev >= 0 ? 1 : firstInit;
            if (b1 == n) { u.mode = t.mode; u.set = -1; u.key = finalKey; }
            else { u.mode = 1; u.set = nAux++; u.key = t.lev[b1 - 1] + 0.5; prev = u.set; }
            list.push_back(u);
            if (b1 == n) break;
        }
    };
    auto flush = [&](std::vector<Tmp>& list) {
        std::stable_sort(list.begin(), list.end(), [](const Tmp& x, const Tmp& y) { return x.key < y.key; });
        for (const Tmp& t : list) {
            out.taskI.push_back(t.I); out.taskJ.push_back(t.J); out.taskMode.push_back((unsigned char)t.mode);
            out.taskWait.push_back(t.wait); out.taskSet.push_back(t.set); out.taskInit.push_back((unsigned char)t.init);
            out.termA.insert(out.termA.end(), t.a.begin(), t.a.end());
            out.termB.insert(out.termB.end(), t.b.begin(), t.b.end());
            out.termPtr.push_back((int64_t)out.termA.size());
        }
        list.clear();
    };
    std::vector<Tmp> list;
    Tmp tmp;
    if (out.nParts > 1 && me >= 0) {
        for (int J : cols) {
            if (out.colOwner[J] != me) continue;
            for (int e = out.colPtr[J]; e < out.colPtr[J + 1]; ++e)
                if (collect(out.slotI[out.colSlot[e]], J, 0, me, tmp)) emit_chain(tmp, false, list);
        }
        for (int J : cols) {
            if (out.colOwner[J] >= 0) continue;
            for (int e = out.colPtr[J]; e < out.colPtr[J + 1]; ++e)
                if (collect(out.slotI[out.colSlot[e]], J, 1, me, tmp)) emit_chain(tmp, false, list);
        }
        flush(list);
    }
    out.nTasks1 = (int)out.taskI.size();
    const bool distributed = out.nParts > 1;
    for (int J : cols) {
        if (out.colOwner[J] >= 0) continue;
        for (int e = out.colPtr[J]; e < out.colPtr[J + 1]; ++e)
            if (collect(out.slotI[out.colSlot[e]], J, 0, -1, tmp)) emit_chain(tmp, distributed, list);   // distributed: the top tiles hold the summed partial results
    }
    flush(list);
    out.nAux = nAux;
    out.nTasks = (int)out.taskI.size();
    out.nTerms = (int64_t)out.termA.size();
    // two queues per phase: the tasks on the dependency chain (every diagonal tile and, per column, the tile in the
    // row of its elimination-tree parent - the last input of the parent's diagonal tile) and the bulk
    out.queue.clear();
    for (int ph = 0; ph < 2; ++ph) {
        const int t0 = ph == 0 ? 0 : out.nTasks1, t1 = ph == 0 ? out.nTasks1 : out.nTasks;
        for (int crit = 1; crit >= 0; --crit) {
            out.qOff[2 * ph + (1 - crit)] = (int)out.queue.size();
            for (int t = t0; t < t1; ++t) {
                const bool c = out.taskMode[t] == 0 && (out.taskI[t] == out.taskJ[t] || out.taskI[t] == parent[out.taskJ[t]]);
                if (c == (crit == 1)) out.queue.push_back(t);
            }
        }
    }
    out.qOff[4] = (int)out.queue.size();
    // backward substitution: top columns (descending level) first, then this part's own columns
    out.bwdCols.clear();
    for (auto it = cols.rbegin(); it != cols.rend(); ++it) if (out.colOwner[*it] < 0) out.bwdCols.push_back(*it);
    out.nBwd1 = (int)out.bwdCols.size();
    for (auto it = cols.rbegin(); it != cols.rend(); ++it) if (out.colOwner[*it] >= 0 && out.colOwner[*it] == me) out.bwdCols.push_back(*it);
    return DBAT_OK;
}

// ---- C entry point for tests and tools (host only, no device needed) ---------------------------------------
// obs_img / obs_op 1-based as in dbat_problem_desc; nEO (nImg) estimated EO elements per image.  Fills
// counts[16] = {nT, ld, nS, nSlots, nSlotsS, nTasks, nTerms, depth, mode, nSeg} and, when the pointers are not
// NULL, imgS (nImg), tix (nT*nT, needs a second call once nT is known), taskIJ (2*nTasks), termPtr (nTasks+1),
// termAB (2*nTerms), level (nT).
static TileSym g_last_sym;
extern "C" int dbat_tile_symbolic(int64_t nImg, int64_t nOP, int64_t nObs, const int64_t* obs_img,
                                  const int64_t* obs_op, const int64_t* nEO, int64_t nIO, int64_t mode,
                                  int64_t leafImages, int64_t* counts) {
    // counts[14], counts[15] on entry: nParts, myPart of a distributed factorisation (0, 0 = one part)
    if (nImg <= 0 || !obs_img || !obs_op || !nEO || !counts) return DBAT_E_BADARG;
    std::vector<int> start((size_t)nOP + 1, 0), imgs((size_t)nObs);
    for (int64_t o = 0; o < nObs; ++o) {
        if (obs_op[o] < 1 || obs_op[o] > nOP || obs_img[o] < 1 || obs_img[o] > nImg) return DBAT_E_BADARG;
        ++start[(size_t)obs_op[o]];
    }
    std::partial_sum(start.begin(), start.end(), start.begin());
    {
        std::vector<int> fill(start.begin(), start.end() - 1);
        for (int64_t o = 0; o < nObs; ++o) imgs[(size_t)fill[(size_t)obs_op[o] - 1]++] = (int)(obs_img[o] - 1);
    }
    std::vector<int64_t> ap; std::vector<int32_t> ad;
    covis_graph((int)nImg, (int)nOP, start.data(), imgs.data(), ap, ad);
    std::vector<int> ne((size_t)nImg);
    for (int64_t i = 0; i < nImg; ++i) ne[(size_t)i] = (int)nEO[i];
    const int nParts = counts[14] > 0 ? (int)counts[14] : 1, myPart = (int)counts[15];
    int rc = tile_symbolic((int)nImg, ap.data(), ad.data(), ne.data(), (int)nIO, (int)mode, (int)leafImages, g_last_sym, nParts, myPart);
    if (rc) return rc;
    const TileSym& s = g_last_sym;
    counts[0] = s.nT; counts[1] = s.ld; counts[2] = s.nS; counts[3] = s.nSlots; counts[4] = s.nSlotsS;
    counts[5] = s.nTasks; counts[6] = s.nTerms; counts[7] = s.depth; counts[8] = s.order_mode; counts[9] = s.nSeg;
    counts[10] = s.ioS; counts[11] = s.nTasks1; counts[12] = s.nTopS; counts[13] = s.nTop; counts[14] = s.nParts; counts[15] = s.nOwnS;
    return DBAT_OK;
}
extern "C" int dbat_tile_symbolic_get(int64_t* imgS, int64_t* tix, int64_t* taskIJ, int64_t* termPtr,
                                      int64_t* termAB, int64_t* level, int64_t* s2kind, int64_t* bwdCols) {
    const TileSym& s = g_last_sym;
    if (s.nT == 0) return DBAT_E_BADARG;
    if (imgS) for (size_t i = 0; i < s.imgS.size(); ++i) imgS[i] = s.imgS[i];
    if (tix) for (size_t i = 0; i < s.tix.size(); ++i) tix[i] = s.tix[i];
    if (taskIJ) for (int t = 0; t < s.nTasks; ++t) { taskIJ[2 * t] = s.taskI[t]; taskIJ[2 * t + 1] = s.taskJ[t]; }
    if (termPtr) for (size_t i = 0; i < s.termPtr.size(); ++i) termPtr[i] = s.termPtr[i];
    if (termAB) for (int64_t t = 0; t < s.nTerms; ++t) { termAB[2 * t] = s.termA[t]; termAB[2 * t + 1] = s.termB[t]; }
    if (level) for (int J = 0; J < s.nT; ++J) level[J] = s.level[J];
    if (s2kind) for (int k = 0; k < s.ld; ++k) s2kind[k] = s.s2kind[k];
    if (bwdCols) { for (int J = 0; J < s.nT; ++J) bwdCols[J] = -1; for (size_t k = 0; k < s.bwdCols.size(); ++k) bwdCols[k] = s.bwdCols[k]; }
    return DBAT_OK;
}
// taskMode (nTasks), colOwner (nT), ownSBegin (nParts+1) of the last analysis
extern "C" int dbat_tile_symbolic_get2(int64_t* taskMode, int64_t* colOwner, int64_t* ownSBegin) {
    const TileSym& s = g_last_sym;
    if (s.nT == 0) return DBAT_E_BADARG;
    // taskMode: 4 values per task: mode, wait (aux flag or -1), set (aux flag or -1), init (1 = start from the tile)
    if (taskMode) for (int t = 0; t < s.nTasks; ++t) {
        taskMode[4 * t] = s.taskMode[t]; taskMode[4 * t + 1] = s.taskWait[t]; taskMode[4 * t + 2] = s.taskSet[t]; taskMode[4 * t + 3] = s.taskInit[t];
    }
    if (colOwner) for (int J = 0; J < s.nT; ++J) colOwner[J] = s.colOwner[J];
    if (ownSBegin) for (size_t k = 0; k < s.ownSBegin.size(); ++k) ownSBegin[k] = s.ownSBegin[k];
    return DBAT_OK;
}
