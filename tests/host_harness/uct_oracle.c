/* uct_oracle.c -- ddz_ref_uct_batch: the batched UCT search of ddz_uct_search (include/ddz_b200.h) restated over the CPU
 * oracle (oracle/ddz_oracle.c: int8 count vectors, ddz_ref_mcts_moves, ddz_ref_get_moves_fast, ddz_ref_philox).
 * TEST INFRASTRUCTURE ONLY: tests/uct_philox_reference.py builds it together with the oracle and compares it with the
 * Python restatement of the algorithm (CPU) and with the device's whole trees (GPU).
 *
 * Written from the contract, not from the kernel: every node keeps its untried entries as an explicit list and pops the
 * i-th one (the reference's list.pop(i), tree.py:42); children are an array in expansion order; playouts re-generate the
 * move list at every decision.  UCB1 and the win rates are evaluated with plain C doubles; build with
 * -ffp-contract=off so that no multiply-add is fused (the device uses correctly rounded operations one by one). */
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#include "../../oracle/ddz_oracle.h"

#define TREE_STEP 0x80000000u

typedef struct {
    int8_t hand[3][15], recent[3][15], move[15];
    int cur, winner, parent, index, visits, wins;
    int nuntried;
    int8_t (*untried)[15];   /* the entries not expanded yet, in list order */
    int nchild;
    int* child;              /* node ids, expansion order */
} node_t;

typedef struct {
    const int8_t* hands; const int8_t* recent; const int32_t* cur; const uint8_t* live;
    int budget, width, prune; double c; uint64_t seed, env0;
    int32_t *choice, *nnodes, *parent, *visits, *wins, *index, *root_n;
    uint64_t *move, *node_move;
    int b0, b1;
} job_t;

static int empty15(const int8_t* a) { for (int r = 0; r < 15; r++) if (a[r]) return 0; return 1; }

/* the trick to beat: the previous player's hand-out, else the one before (envi.py:103-110) */
static const int8_t* trick(const int8_t recent[3][15], int cur) {
    const int8_t* p = recent[(cur + 2) % 3];
    return empty15(p) ? recent[(cur + 1) % 3] : p;
}

/* the node's entries: the bot's pruned list or the canonical list */
static int entries(const int8_t hand[15], const int8_t last[15], int prune, int8_t out[][15]) {
    return prune ? ddz_ref_mcts_moves(hand, last, &out[0][0], DDZ_REF_MAX_LEGAL)
                 : ddz_ref_get_moves_fast(hand, last, &out[0][0], DDZ_REF_MAX_LEGAL);
}

static int won(int winner, int me) { return (winner == 1) == (me == 1); }

/* one random playout to the end of the game from (hand, recent, cur); 1 if the searching side won */
static int playout(const node_t* x, int prune, uint64_t seed, uint64_t stream, int me) {
    int8_t hand[3][15], recent[3][15], list[DDZ_REF_MAX_LEGAL][15];
    memcpy(hand, x->hand, sizeof hand);
    memcpy(recent, x->recent, sizeof recent);
    int cur = x->cur;
    for (uint32_t t = 0;; t++) {
        const int n = entries(hand[cur], trick((const int8_t(*)[15])recent, cur), prune, list);
        const int8_t* mv = list[ddz_ref_philox(seed, stream, t) % (uint32_t)n];
        for (int r = 0; r < 15; r++) hand[cur][r] -= mv[r];
        memcpy(recent[cur], mv, 15);
        if (!empty15(mv) && empty15(hand[cur])) return won(cur, me);
        cur = (cur + 1) % 3;
    }
}

static void search_root(const job_t* j, int b) {
    const int budget = j->budget, W = j->width, me = j->cur[b];
    node_t* T = (node_t*)calloc((size_t)budget + 1, sizeof(node_t));
    int8_t list[DDZ_REF_MAX_LEGAL][15];
    uint32_t draws = 0;
    const uint64_t env = j->env0 + (uint64_t)b;
    int nn = 0;
#define NEW_NODE(id, src_hand, src_recent, cur_, winner_, parent_, index_)                                   \
    do {                                                                                                    \
        node_t* y_ = &T[id];                                                                                \
        memcpy(y_->hand, src_hand, sizeof y_->hand); memcpy(y_->recent, src_recent, sizeof y_->recent);     \
        y_->cur = (cur_); y_->winner = (winner_); y_->parent = (parent_); y_->index = (index_);             \
        if (y_->winner < 0) {                                                                               \
            const int n_ = entries(y_->hand[y_->cur], trick((const int8_t(*)[15])y_->recent, y_->cur), j->prune, list); \
            y_->untried = malloc((size_t)(n_ ? n_ : 1) * 15); memcpy(y_->untried, list, (size_t)n_ * 15);   \
            y_->nuntried = n_;                                                                              \
        }                                                                                                   \
        y_->child = malloc((size_t)DDZ_REF_MAX_LEGAL * sizeof(int));                                        \
    } while (0)
    const int8_t* h0 = j->hands + (size_t)b * 45;
    const int8_t* r0 = j->recent + (size_t)b * 45;
    NEW_NODE(0, h0, r0, me, -1, -1, -1);
    nn = 1;
    if (!j->live[b] || T[0].nuntried == 0) {
        j->choice[b] = -1; j->move[b] = ~0ull; j->root_n[b] = 0; j->nnodes[b] = 0;
        free(T[0].untried); free(T[0].child); free(T);
        return;
    }
    for (int it = 0; it < budget; it++) {
        int x = 0;
        while (T[x].winner < 0) {                                  /* tree policy */
            node_t* X = &T[x];
            if (X->nuntried > 0) {                                 /* expand the i-th remaining entry */
                const int i = (int)(ddz_ref_philox(j->seed, env, TREE_STEP + draws++) % (uint32_t)X->nuntried);
                int8_t mv[15];
                memcpy(mv, X->untried[i], 15);
                memmove(X->untried[i], X->untried[i + 1], (size_t)(X->nuntried - i - 1) * 15);
                X->nuntried--;
                const int8_t* last = trick((const int8_t(*)[15])X->recent, X->cur);
                const int nfull = ddz_ref_get_moves_fast(X->hand[X->cur], last, &list[0][0], DDZ_REF_MAX_LEGAL);
                int index = -1;
                for (int k = 0; k < nfull && index < 0; k++) if (!memcmp(list[k], mv, 15)) index = k;
                int8_t hand[3][15], recent[3][15];
                memcpy(hand, X->hand, sizeof hand); memcpy(recent, X->recent, sizeof recent);
                for (int r = 0; r < 15; r++) hand[X->cur][r] -= mv[r];
                memcpy(recent[X->cur], mv, 15);
                const int winner = (!empty15(mv) && empty15(hand[X->cur])) ? X->cur : -1;
                NEW_NODE(nn, hand, recent, (X->cur + 1) % 3, winner, x, index);
                memcpy(T[nn].move, mv, 15);
                X->child[X->nchild++] = nn;
                x = nn++;
                break;
            }
            /* UCB1: the maximum for the searching player, the minimum for the others; a random one among exact ties */
            const double lnN = log((double)X->visits);
            double v[DDZ_REF_MAX_LEGAL], target = 0;
            for (int k = 0; k < X->nchild; k++) {
                const node_t* ch = &T[X->child[k]];
                v[k] = (double)ch->wins / (double)ch->visits + j->c * sqrt(2.0 * lnN / (double)ch->visits);
                if (k == 0 || (X->cur == me ? v[k] > target : v[k] < target)) target = v[k];
            }
            int tied[DDZ_REF_MAX_LEGAL], nt = 0;
            for (int k = 0; k < X->nchild; k++) if (v[k] == target) tied[nt++] = X->child[k];
            x = nt == 1 ? tied[0] : tied[ddz_ref_philox(j->seed, env, TREE_STEP + draws++) % (uint32_t)nt];
        }
        int reward = 0;                                            /* default policy */
        if (T[x].winner >= 0) reward = W * won(T[x].winner, me);
        else
            for (int w = 0; w < W; w++)
                reward += playout(&T[x], j->prune, j->seed, ((env * (uint64_t)budget) + (uint64_t)it) * (uint64_t)W + (uint64_t)w, me);
        for (int y = x; y >= 0; y = T[y].parent) { T[y].visits += W; T[y].wins += reward; }   /* back-up */
    }
    /* answer: the root child with the best wins / visits, a random one among exact ties */
    const node_t* R = &T[0];
    double best = 0;
    for (int k = 0; k < R->nchild; k++) {
        const double r = (double)T[R->child[k]].wins / (double)T[R->child[k]].visits;
        if (k == 0 || r > best) best = r;
    }
    int tied[DDZ_REF_MAX_LEGAL], nt = 0;
    for (int k = 0; k < R->nchild; k++)
        if ((double)T[R->child[k]].wins / (double)T[R->child[k]].visits == best) tied[nt++] = R->child[k];
    const int pick = nt == 1 ? tied[0] : tied[ddz_ref_philox(j->seed, env, TREE_STEP + draws++) % (uint32_t)nt];
    j->choice[b] = T[pick].index;
    j->move[b] = ddz_ref_pack(T[pick].move);
    j->root_n[b] = R->nchild;
    j->nnodes[b] = nn;
    const size_t o = (size_t)b * (size_t)(budget + 1);
    for (int k = 0; k < nn; k++) {
        j->parent[o + k] = T[k].parent; j->visits[o + k] = T[k].visits; j->wins[o + k] = T[k].wins;
        j->index[o + k] = T[k].index; j->node_move[o + k] = ddz_ref_pack(T[k].move);
    }
    for (int k = 0; k < nn; k++) { free(T[k].untried); free(T[k].child); }
    free(T);
#undef NEW_NODE
}

static void* worker(void* p) {
    const job_t* j = (const job_t*)p;
    for (int b = j->b0; b < j->b1; b++) search_root(j, b);
    return 0;
}

/* B roots (hands / recent int8 [B][3][15], cur int32 [B], live uint8 [B]) on nthreads host threads.  Outputs: choice,
 * move (~0 for a root that is not searched), root_n, nnodes [B]; per node [B][budget + 1] in creation order: parent,
 * visits, wins, index (of the move in the parent's canonical list), node_move (packed; root 0).  The root children are
 * nodes 1 .. root_n. */
int ddz_ref_uct_batch(const int8_t* hands, const int8_t* recent, const int32_t* cur, const uint8_t* live, int B, int budget,
                      int width, int prune, double c, uint64_t seed, uint64_t env0, int nthreads, int32_t* choice,
                      uint64_t* move, int32_t* root_n, int32_t* nnodes, int32_t* parent, int32_t* visits, int32_t* wins,
                      int32_t* index, uint64_t* node_move) {
    if (B <= 0 || budget < 1 || width < 1) return -1;
    if (nthreads < 1) nthreads = 1;
    if (nthreads > B) nthreads = B;
    job_t* jobs = (job_t*)calloc((size_t)nthreads, sizeof(job_t));
    pthread_t* th = (pthread_t*)calloc((size_t)nthreads, sizeof(pthread_t));
    for (int i = 0; i < nthreads; i++) {
        job_t* j = &jobs[i];
        j->hands = hands; j->recent = recent; j->cur = cur; j->live = live;
        j->budget = budget; j->width = width; j->prune = prune; j->c = c; j->seed = seed; j->env0 = env0;
        j->choice = choice; j->move = move; j->root_n = root_n; j->nnodes = nnodes; j->parent = parent;
        j->visits = visits; j->wins = wins; j->index = index; j->node_move = node_move;
        j->b0 = (int)((int64_t)B * i / nthreads); j->b1 = (int)((int64_t)B * (i + 1) / nthreads);
        pthread_create(&th[i], 0, worker, j);
    }
    for (int i = 0; i < nthreads; i++) pthread_join(th[i], 0);
    free(jobs); free(th);
    return 0;
}
