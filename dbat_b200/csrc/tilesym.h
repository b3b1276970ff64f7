// tilesym.h — host-side symbolic analysis of the reduced camera system for the sparse tile Cholesky
// (tilechol.cu).  SURVEY.md §8(f) N4: the reference factors the camera block densely
// (code/bundle/bundle_cov.m:97); its ordering experiments are code/bundle/private/blkcolperm.m and
// code/test/postcov/reorder_test.m.  Here the images are ordered by nested dissection (or reverse
// Cuthill-McKee) on the co-visibility graph, the shared IO block and the right-hand side come last
// ([OP; EO; IO] as in bundle_cov.m:76-84), and the factorisation works on 64 x 64 tiles of the
// resulting sparse pattern.
#pragma once
#include <cstdint>
#include <vector>

#define TC_T 64                    // tile size
#define TC_TT (TC_T * TC_T)

struct TileSym {
    int nT = 0;                    // tile rows / columns
    int ld = 0;                    // order of the padded system = nT * TC_T; the last row carries the rhs
    int nS = 0;                    // number of real unknowns in S (EO + IO columns)
    // stored tiles.  Slot order: [top S | top fill | owned-by-part-0 S | ... | owned-by-part-(nParts-1) S | owned fill ...]
    // ("top" = tile columns every rank factors; with one part everything is top).  nSlotsS counts the tiles of
    // the pattern of S itself: the ranges [0, nTopS) and [nTop, nTop + nOwnS).
    int nSlots = 0, nSlotsS = 0;
    int nTopS = 0, nTop = 0, nOwnS = 0;
    int nParts = 1, myPart = 0;
    std::vector<int> ownSBegin;    // nParts + 1: slot range of the S tiles owned by every part
    std::vector<int> colOwner;     // per tile column: owning part, -1 = top
    int nTasks = 0, nTasks1 = 0, depth = 0;   // tasks [0, nTasks1): phase 1 (own columns + partial sums into top tiles),
                                              // [nTasks1, nTasks): phase 2 (top columns, after the partial sums are reduced)
    std::vector<unsigned char> taskMode;      // 0 = final (factor / solve, sets the tile's flag), 1 = partial sum only
    std::vector<int> taskWait, taskSet;       // chains of partial sums on one tile: auxiliary flag to wait for / to set (-1: none)
    std::vector<unsigned char> taskInit;      // 1: the accumulation starts from the tile's content, 0: from zero
    int nAux = 0;
    std::vector<int> queue;                   // task ids: [phase 1 chain | phase 1 bulk | phase 2 chain | phase 2 bulk]
    int qOff[5] = {0, 0, 0, 0, 0};
    int nBwd1 = 0;                            // bwdCols[0, nBwd1): top columns; [nBwd1, ..): this part's own columns
    int64_t nTerms = 0;
    int order_mode = 0;            // 0 natural, 1 rcm, 2 nested dissection
    int nSeg = 0;
    std::vector<int> imgOrder;     // image ids in elimination order
    std::vector<int> imgRank;      // inverse of imgOrder
    std::vector<int> imgS;         // per image id: S index of its first estimated EO column (-1: none)
    int ioS = 0;                   // S index of the first estimated shared IO column
    std::vector<int> s2kind;       // per S index: 0 padding (identity), 1 unknown, 2 rhs row
    std::vector<int> tix;          // nT x nT (row-major, [I * nT + J], I >= J): slot or -1
    std::vector<int> slotI, slotJ; // tile coordinates of every slot
    std::vector<int> colPtr, colSlot;   // per tile column: its slots, rows ascending (the diagonal tile first)
    std::vector<int> taskI, taskJ;      // task list in execution (= priority) order
    std::vector<int64_t> termPtr;       // nTasks + 1
    std::vector<int> termA, termB;      // slots of L(I,k), L(J,k) for every term of every task
    std::vector<int> level;             // elimination-tree level of every tile column
    std::vector<int> bwdCols;           // tile columns for the backward substitution (descending level)
};

// adjacency of the co-visibility graph in CSR form (no self loops needed); nEO[i] = number of estimated
// EO elements of image i (0..6); nIO = number of estimated shared IO columns.
// mode: 0 natural, 1 rcm, 2 nested dissection, -1 automatic.
// nParts / myPart: distributed factorisation - the elimination tree is cut into nParts (a power of two) subtrees,
// part g factors the columns of subtree g, everybody the separators above the cut (nParts = 1: everything local).
int tile_symbolic(int nImg, const int64_t* adjPtr, const int32_t* adj, const int* nEO, int nIO, int mode,
                  int leafImages, TileSym& out, int nParts = 1, int myPart = 0);

// co-visibility graph from (0-based) point-major image lists
void covis_graph(int nImg, int nOP, const int* pt_start, const int* img_pm, std::vector<int64_t>& adjPtr,
                 std::vector<int32_t>& adj);
