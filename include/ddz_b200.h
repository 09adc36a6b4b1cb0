/*
 * ddz_b200.h -- C-ABI of the B200-native batched Doudizhu environment (libddz_b200.so).
 *
 * This is the drop-in boundary for the rollout path of charleschen003/doudizhu-rl.  It replaces the two
 * pre-compiled native modules the reference loads from precompiled/ (reference envi.py:10-13):
 *   `env`  (class env.Env: reset / prepare / step_manual / get_* / get_state_prob)   and
 *   `r`    (r.get_moves(hand15, last15))
 * plus the per-decision Python loops of envi.py that sit directly on them (face, valid_actions,
 * batch_arr2onehot, _update).  Every entry point below cites the reference interface it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named host_*;
 *   - the caller (PyTorch) owns every buffer the launchers touch, and no launcher keeps a pointer after it returns.
 *     Two opt-in helpers do own resources: ddz_pipe_* / ddz_mpipe_* objects hold CUDA streams and events (and remember
 *     the destination of a staged deal-pool upload until it is committed), and ddz_rows_alloc maps compressible device
 *     memory that the caller frees with ddz_rows_free;
 *   - all launches are asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default);
 *   - return value: 0 ok, <0 error (DDZ_E_*); no exceptions, nothing printed;
 *   - there is NO CPU fallback: without a CUDA device every launcher returns DDZ_E_CUDA.
 *
 * Data formats
 *   counts   a hand / move / history is 15 per-rank counts, rank 0='3' ... 11='A', 12='2', 13=black joker,
 *            14=red joker (reference config.py:16-18, envi.py:119-137), packed 4 bits per rank into a
 *            uint64 (rank r in bits [4r, 4r+4)); a pass is 0.
 *   state    opaque, ddz_state_bytes(B) bytes, 8-byte aligned, struct-of-arrays:
 *            uint64 hand[3][B], hist[3][B], recent[3][B]  (role 0=up, 1=lord, 2=down, envi.py:24)
 *            uint32 meta[B]: bits 0-1 role to move, bit 2 done, bits 3-4 winner, bit 5 sticky error,
 *            bits 8-31 deals consumed.
 *   legal    CSR: offsets int32[B+1], actions_u64[offsets[B]] packed counts in canonical order
 *            (card.py action-space order, pass first when following), actions_f32[offsets[B]][15][4]
 *            thermometer one-hot (envi.py:140-146), face float32[B][C][15][4] (envi.py:87-217).
 *   stats    int64[16], accumulated (never cleared by the library):
 *            0 games finished, 1 lord wins, 2 down wins, 3 up wins, 4 env-steps applied,
 *            5 sum lord reward, 6 sum farmer reward (down+up), 7 errors, 8 legal moves emitted, 9 passes.
 */
#ifndef DDZ_B200_H
#define DDZ_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDZ_ABI_VERSION 3   /* 3: ddz_mcts_moves, ddz_playout_pruned, ddz_q_features (+ ddz_uct_search, ddz_uct_workspace_bytes,
                            * ddz_determinize, ddz_uct_pool, ddz_encode_face_gather, ddz_move_ids, ddz_moves_of_ids, ddz_legal_mask:
                            * new entry points only, backward compatible).  2: ddz_mpipe_*, ddz_set_tile_order, ddz_prob_form; cut lists are played
                            * from their visible part */
#define DDZ_MAX_LEGAL 512  /* upper bound of legal moves of one decision (worst known hand: 497) */

#define DDZ_E_ARG -1     /* bad argument (NULL pointer, B <= 0, unknown variant/mode) */
#define DDZ_E_CUDA -2    /* CUDA runtime error / no device */

/* face variants = the reference's four Env classes */
#define DDZ_FACE_FIRST 0          /* envi.py:87-96    Env                     C=4 */
#define DDZ_FACE_COMPLICATED 1    /* envi.py:165-178  EnvComplicated          C=7 */
#define DDZ_FACE_COOPERATION 2    /* envi.py:182-198  EnvCooperation          C=9 */
#define DDZ_FACE_SIMPLIFY 3       /* envi.py:202-217  EnvCooperationSimplify  C=6 */

/* how ddz_step / ddz_rollout_step pick the move of env b out of its N legal moves */
#define DDZ_CHOICE_INDEX 0   /* choice[b] is the index (dqn.py:60,70 argmax / randint)                    */
#define DDZ_CHOICE_MOD 1     /* (uint32)choice[b] % N  -- host-supplied entropy, envi.py:83 random.choice */
#define DDZ_CHOICE_PHILOX 2  /* philox4x32-10(key=seed, ctr=(env0+b, stepno)) % N, no input buffer        */
#define DDZ_CHOICE_MOVE 3    /* moves[b] is the packed move itself (envi.py:63-70 step_manual); must be legal */

/* stepno value for ddz_rollout_step: take the Philox step number from the counter kept in the workspace (uint32 at
 * byte 12; every stepping launch leaves it at its step number + 1).  Makes a captured CUDA graph replayable. */
#define DDZ_STEPNO_AUTO 0xFFFFFFFFu

int ddz_abi_version(void);
/* layout of the two probability planes of a face (get_state_prob, envi.py:94; get_state_prob_manual, server/core.py:26-33),
 * a build-time choice because nothing in the reference pins it (oracle/SEMANTICS.md): 0 = form A, thermometer of the
 * unknown count (default); 1 = form B, deck60 - known60 element-wise (library built with -DDDZ_PROB_FORM_B) */
int ddz_prob_form(void);
/* How the list-producing launches (observe / rollout_step) hand their 32-env tiles to warps.  DDZ_TILES_AUTO (default):
 * by launch position when the whole grid fits on the device at once (saves an atomic round trip before the first load),
 * else by an atomic ticket in start order.  DDZ_TILES_TICKET: always by ticket -- ask for it when OTHER kernels (a Q-network,
 * a collective) share the GPU with the env launches, so that nothing depends on the grid being co-resident.  Process-wide;
 * returns the previous mode. */
#define DDZ_TILES_AUTO 0
#define DDZ_TILES_TICKET 1
int ddz_set_tile_order(int mode);
int ddz_face_channels(int variant);          /* 4 / 7 / 9 / 6, or DDZ_E_ARG */
size_t ddz_state_bytes(int B);
/* Scratch for observe / rollout_step / legal_moves (n <= B): tile ticket + one look-back word per 32-env tile.
 * The caller zero-fills it ONCE after allocation; every launch re-arms it.  One workspace per stream:
 * two launches that share a workspace must not run concurrently. */
size_t ddz_workspace_bytes(int B);
const char* ddz_last_error(void);            /* text of the last CUDA error seen by this thread */

/* env.Env.reset() + prepare()  (envi.py:30-36, game.py:170-171) with host-chosen shuffles (SURVEY C2):
 * perm int8[pool_games][B][54] card ids (0..51 -> rank id/4, 52/53 jokers), lord_pile int8[pool_games][B]
 * (may be NULL = 0).  Env b takes row (deals_consumed % pool_games)*B + b.  only_done != 0 re-deals only
 * finished envs.  Piles perm[0:17],[17:34],[34:51], bottom [51:54]; pile lord_pile(+bottom) -> lord,
 * next pile -> down, next -> up; lord to move. */
int ddz_reset(void* state, const int8_t* perm, const int8_t* lord_pile, int pool_games, int only_done,
              int64_t* stats, int B, void* stream);

/* env.face + env.valid_actions() for all envs  (envi.py:87-116; r.get_moves envi.py:111;
 * get_state_prob envi.py:94; batch_arr2onehot envi.py:140-146).
 * offsets int32[B+1] and actions_u64[cap] are required; actions_f32 / face may be NULL (skipped).
 * Finished envs have no legal move.  If the total exceeds cap the tail is dropped and stats[7] is bumped; the offsets
 * are still those of the complete lists.  Nothing is read or written out of bounds and no env is lost: the fused step
 * plays a cut list from its visible part, an env whose list was dropped altogether sits that step out (stats[7] counts
 * it, no sticky error) and moves again as soon as a list of its own fits -- or observe again with a larger cap.
 * cap = 0 is valid: only the offsets (and the face) are written, and a fused step from such lists moves no env. */
int ddz_observe(const void* state, void* workspace, int variant, int32_t* offsets, uint64_t* actions_u64,
                float* actions_f32, int64_t cap, float* face, int64_t* stats, int B, void* stream);

/* The two halves of env.valid_actions() on their own (r.get_moves, envi.py:111): the number of legal moves of the player
 * to move in every env in closed form (no list, no workspace; finished envs: 0), and the packed CSR lists without any
 * float tensor (= ddz_observe with actions_f32 = face = NULL).  counts[b] == offsets[b+1] - offsets[b]. */
int ddz_legal_count(const void* state, int32_t* counts, int B, void* stream);
int ddz_legal_emit(const void* state, void* workspace, int32_t* offsets, uint64_t* actions_u64, int64_t cap,
                   int64_t* stats, int B, void* stream);

/* env.step_manual / step_random for all envs  (envi.py:63-70, 79-85, _update :38-43; terminal + sign
 * rule_based/rule_play.py:14-28; rewards game.py:109-118 with magnitudes rewards[role]).
 * offsets/actions_u64 must be the COMPLETE lists ddz_observe produced for the CURRENT state (no overflow: stats[7]).
 * Outputs (any may be NULL): r int8[B] (-1 lord won, +1 farmers won, 0), done uint8[B], cat int8[B]
 * (card.py:13-28 category of the move, -1 if nothing was applied), reward float32[B][3].
 * Finished envs and illegal choices are no-ops (illegal: sticky error bit + stats[7]). */
int ddz_step(void* state, const int32_t* offsets, const uint64_t* actions_u64, const void* choice,
             int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno, const int32_t rewards[3],
             int8_t* r, uint8_t* done, int8_t* cat, float* reward, int64_t* stats, int B, void* stream);

/* One fused env-step = ddz_step, then ddz_reset(only_done=1) when perm != NULL, then ddz_observe of the
 * new state, in ONE launch.  prev_* are the lists of the state being stepped, out_* receive the new
 * lists (ping-pong; they must not alias -- the action lists may when cap = 0 -- and both hold cap moves: of a list that an
 * overflow cut off only the stored part can be chosen from, never an out-of-bounds read; at cap = 0 every live env sits
 * the step out). */
int ddz_rollout_step(void* state, void* workspace, int variant,
                     const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                     const void* choice, int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno,
                     const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                     int8_t* r, uint8_t* done, int8_t* cat, float* reward,
                     int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                     float* face, int64_t* stats, int B, void* stream);

/* nsteps consecutive ddz_rollout_step's of a policy that needs no host decision in between -- the random rollout of
 * envi.py:79-85 / game.py:259-275 -- enqueued by ONE call, every step's observation kept (a trajectory):
 *   prev_* are the lists of the state the first step starts from;
 *   choice_mode DDZ_CHOICE_PHILOX (choice == NULL) or DDZ_CHOICE_MOD (choice = uint32 [nsteps][B] entropy);
 *   r / done / cat are [nsteps][B], reward [nsteps][B][3] (any may be NULL);
 *   out_offsets int32 [nsteps][B+1], out_actions_u64 [nsteps][cap], out_actions_f32 [nsteps][cap][15][4],
 *   face float32 [nsteps][B][C][15][4]: slice s is the observation after step s (Philox step number stepno + s).
 * nsteps launches of the fused kernel on `stream`, slice s-1 feeding step s.  (A single launch that pipelines the steps
 * as a wavefront was built and measured slower: DESIGN.md 4, profiles/experiments/.) */
int ddz_rollout_steps(void* state, void* workspace, int variant, int nsteps,
                      const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                      const void* choice, int choice_mode, uint64_t seed, uint64_t env0, uint32_t stepno,
                      const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                      int8_t* r, uint8_t* done, int8_t* cat, float* reward,
                      int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                      float* face, int64_t* stats, int B, void* stream);

/* r.get_moves(hand15, last15) for n independent (hand, last) pairs  (envi.py:111, server/core.py:65):
 * hands/lasts packed uint64[n]; last == 0 means lead.  Same CSR outputs as ddz_observe. */
int ddz_legal_moves(const uint64_t* hands, const uint64_t* lasts, void* workspace, int32_t* offsets,
                    uint64_t* actions_u64, int64_t cap, int64_t* stats, int n, void* stream);

/* idx[i]-th move of r.get_moves(hands[i], lasts[i]) in closed form, without building the list (moves[i] = ~0 when idx is
 * out of range); counts (optional) = the list lengths. */
int ddz_kth_moves(const uint64_t* hands, const uint64_t* lasts, const int32_t* idx, uint64_t* moves, int32_t* counts,
                  int n, void* stream);

/* Random playout = the default policy of the reference's MCTS (server/mcts/default_policy.py:4-10, random legal moves
 * until the game ends): plays every env forward for up to max_steps decisions (or to its end), move number
 * philox(seed, env0+b, stepno0+t) % N each time -- exactly what max_steps calls of ddz_rollout_step(DDZ_CHOICE_PHILOX)
 * without re-deal would do, but with no lists or features written.  steps_taken int32[B] may be NULL. */
int ddz_playout(void* state, int max_steps, uint64_t seed, uint64_t env0, uint32_t stepno0, const int32_t rewards[3],
                int32_t* steps_taken, int64_t* stats, int B, void* stream);

/* The first layer of the reference's Q-networks for every legal move, from the packed state and lists (net.py:65-139, the
 * NetComplicated family: four (1,k) convolutions with stride (1,4), max-pool, the (15,1) "shunzi" convolution, net.py:91-97):
 * out[row] = [15 x W | W x 4]: the numbers net.py:99 feeds fc1, the rank features RANK-MAJOR (index r * W + o where net.py:93
 * has o * 15 + r: permute fc1's columns once), the line features as net.py has them (o * 4 + j) -- WITHOUT building the
 * [n, C+1, 15, 4] input of net.py:87-90.
 * Every input plane is a function of one nibble per rank, so the convolutions are sums of table rows:
 * rank_tables float32 [C+1][16][W][4] (T[c][nibble][o][k] = sum_{j<=k} W_k+1[o,c,0,j] * slot_j(nibble); the row of nibble 0
 * must be zero), rank_bias [W][4], line_weights [C+1][15][W], line_bias [W] and out, all 16-byte aligned (rows are
 * stored as float4 / 4 x bfloat16); W = width <= 256, a multiple of 4 (the reference: 256).  Rows and masks as in
 * ddz_encode_state_actions; only the envs [env_begin, env_begin + env_count) are processed and row_base is subtracted from
 * their row numbers (chunking).  out_bf16 != 0: rows are written as bfloat16.  Form-B builds read the form-B nibbles. */
int ddz_q_features(const void* state, int variant, const int32_t* offsets, const uint64_t* actions_u64,
                   const uint8_t* env_mask, const int32_t* dst_offsets, int env_begin, int env_count, int64_t row_base,
                   const float* rank_tables, const float* rank_bias, const float* line_weights, const float* line_bias,
                   int width, void* out, int out_bf16, int B, void* stream);

/* The search bot's own move list and default policy (server/mcts/get_moves.py:36-69, which tree.py:33,86 calls for the
 * tree AND for every playout move): a list of more than 10 moves loses its rocket-kicker moves (:22-34,:56-57), the rest is
 * ranked by  cards_value[move] - 0.1 * cards left in hand  (server/mcts/evaluator.py:17-57, stable sort) and the list
 * becomes  lowest, highest, 2nd lowest, 2nd highest, ...  for int(N/3 + 1) rounds.
 * ddz_mcts_moves: that list for n (hand, last) pairs; moves uint64[n][DDZ_MCTS_MAX_MOVES], counts int32[n].
 * ddz_playout_pruned: ddz_playout drawing entry  philox(...) % len(pruned list)  of that list at every decision. */
#define DDZ_MCTS_MAX_MOVES 344   /* 2 * (DDZ_MAX_LEGAL / 3 + 1), rounded up to a multiple of 8 */
int ddz_mcts_moves(const uint64_t* hands, const uint64_t* lasts, uint64_t* moves, int32_t* counts, int n, void* stream);
int ddz_playout_pruned(void* state, int max_steps, uint64_t seed, uint64_t env0, uint32_t stepno0, const int32_t rewards[3],
                       int32_t* steps_taken, int64_t* stats, int B, void* stream);

/* The search bot itself (server/mcts/interface.py:37-45) for B positions in ONE launch: `budget` iterations of UCT
 * (tree policy: walk down while a node is fully expanded by UCB1 -- the maximum where the node's player is the searching
 * player, the minimum elsewhere, partner farmer included --, expand one untried entry at the first node that has one;
 * default policy: `width` random playouts to the end, = ddz_playout_pruned / ddz_playout, or width x won for a node whose
 * move ended the game; back-up: visits += width, wins += playouts the searching side won), then the root child with the
 * best wins / visits.  Root b is env b of `state` (read only): the searching player is the role to move, the trick to
 * beat the previous hand-out (else the one before), hist is not used.  A node's entries are the bot's pruned list
 * (ddz_mcts_moves order, duplicates are separate entries) when prune != 0, else the canonical list; the expanded entry is
 * the i-th REMAINING untried entry in list order (list.pop(i)).
 * Draws (Philox, as ddz_playout):
 *   tree draw j of root b = philox(seed, env0 + b, 0x80000000 + j): j counts every expansion draw (u % remaining, taken even
 *   when one entry remains) and every tie draw among k >= 2 exactly equal UCB / final values (u % k over the tied
 *   children in expansion order), in the order they happen;
 *   playout w of iteration it of root b = philox(seed, ((env0 + b) * budget + it) * width + w, t) at its decision t.
 * UCB1 = wins / visits + c * sqrt(2 * ln_table[visits of the parent] / visits) in double, correctly rounded operations,
 * no contraction; ln_table is device double[budget * width + 1], ln_table[n] = log((double)n) of the host C library.
 * Outputs: choice int32[B] = index of the chosen move in the env's canonical legal list (feeds ddz_step /
 * ddz_rollout_step with DDZ_CHOICE_INDEX), -1 for an env that is masked out (env_mask uint8[B] or NULL = all), finished or
 * without a move; move uint64[B] (optional) = the packed move, or ~0.  Root table (optional; root_n NULL skips it):
 * root_n int32[B] = number of root children, and for the first min(root_n, root_stride) of them in expansion order
 * root_moves uint64 / root_visits int32 / root_wins int32 [B][root_stride].  Masked-out and finished roots take no draw,
 * so they never shift another root's search; env0 chunks a batch (two calls over halves with their env0 = one call).
 * Bounds: 1 <= budget <= DDZ_UCT_MAX_BUDGET, 1 <= width <= DDZ_UCT_MAX_WIDTH, budget * width <= DDZ_UCT_MAX_PLAYOUTS, c
 * finite; else (or NULL state / workspace / ln_table / choice, B <= 0) DDZ_E_ARG before any CUDA call.
 * Workspace (no zero-fill needed; one per concurrent launch), ddz_uct_workspace_bytes(B, budget) =
 *   round_up(4 B, 256) + B (budget + 1) DDZ_UCT_NODE_BYTES  (0 for arguments out of range): int32 nnodes[B] (0 for a root
 * that was not searched), then from byte round_up(4 B, 256) the tree of root b at node b * (budget + 1): node 0 is the
 * root, node k the k-th one created (expansion order); a node's children are the nodes whose parent it is.  Node, 160 bytes:
 *   0 uint32 untried[16] (bit j: entry j not expanded)   64 uint64 hand[3]   88 uint64 recent[3]
 *   112 uint64 move (root 0)   120 int32 parent (root -1)   124 int32 first_child   128 int32 last_child (-1 / -1: none)
 *   132 int32 nchild   136 int32 visits   140 int32 wins   144 int16 nentries   146 int16 remaining
 *   148 int16 index (of move in the parent's canonical list; root -1)   150 int8 cur   151 int8 winner (-1: none)   152 pad */
#define DDZ_UCT_MAX_BUDGET 65536
#define DDZ_UCT_MAX_WIDTH 1024
#define DDZ_UCT_MAX_PLAYOUTS (1 << 24)   /* budget * width */
#define DDZ_UCT_NODE_BYTES 160
size_t ddz_uct_workspace_bytes(int B, int budget);
int ddz_uct_search(const void* state, const uint8_t* env_mask, void* workspace, int budget, int width, int prune, double c,
                   const double* ln_table, uint64_t seed, uint64_t env0, int32_t* choice, uint64_t* move,
                   int32_t* root_n, uint64_t* root_moves, int32_t* root_visits, int32_t* root_wins, int root_stride,
                   int B, void* stream);

/* Search from the player's own view (determinized UCT, perfect-information Monte Carlo): sample D complete deals that agree
 * with what the player to move has seen, search each with ddz_uct_search, add up the root statistics per move.
 *
 * ddz_determinize: out_state holds ddz_state_bytes(B * D) bytes; env b * D + d is determinization d of env b.  The mover's
 * hand (role m = meta bits 0-1), hist[3], recent[3] and meta are copied from env b; the hands of roles a = (m+1)%3 and
 * c = (m+2)%3 become a random split of the UNSEEN cards = full deck - hand[m] - hist[0] - hist[1] - hist[2], a getting as
 * many cards as its hand holds and c the rest.  Draw rule: the unseen cards are walked in rank order 0..14, one physical
 * card at a time, j = 0 .. U-1; card j goes to a when
 *     philox(seed, (env0 + b) * D + d, 0xC0000000 + j) % (ra + rc) < ra
 * (ra, rc: the slots still open in each hand), else to c; a draw is taken for every card, also when one side is full.
 * This is selection sampling: every split of the (distinguishable) unseen cards into those two sizes is equally likely, up
 * to the modulo bias of a 32-bit draw.  The Philox stream (seed, (env0 + b) * D + d) is the one ddz_uct_search uses for
 * that determinization when it is called with env0' = (env0 + b0) * D over the B * D envs; the ranges cannot collide:
 * determinization draws take steps 0xC0000000 .. +36, tree draws start at 0x80000000 and a tree takes fewer than 2^30 of
 * them, playouts take steps below 400.
 * Masked-out (env_mask uint8[B], NULL = all) and finished envs are copied unchanged and take no draw.  A root whose view no
 * deal agrees with (a negative unseen count for a rank, or U != |hand[a]| + |hand[c]|, e.g. a full-information env with
 * zero hist) is copied with meta bits 2 (done) and 5 (sticky error) set in all D copies, and stats[7] (stats may be NULL)
 * counts it once; the search then skips those copies as finished.
 * NULL state / out_state, B <= 0, D outside 1..DDZ_PIMC_MAX_DETERMINIZATIONS or B * D > INT_MAX: DDZ_E_ARG before any CUDA
 * call.
 *
 * ddz_uct_pool: `workspace` as written by ddz_uct_search over B * D roots (tree b * D + d, same budget).  For root b, the
 * root children (parent 0) of every tree with nnodes > 0 add their visits and wins under their canonical `index`
 * (duplicate pruned entries of one tree add up too): pooled_visits / pooled_wins int32 [B][DDZ_MAX_LEGAL] (optional, each
 * may be NULL), in the order of the env's canonical legal list.  choice[b] = the index with the best pooled wins / visits
 * among those with visits > 0 (W_i * V_j against W_j * V_i in 64 bits; exact ties go to the LOWEST index), -1 when no tree
 * of b was searched; move[b] (optional) = the packed move at that index (select_legal over the root's hand and trick), or
 * ~0.  NULL workspace / choice, B <= 0, budget outside 1..DDZ_UCT_MAX_BUDGET, D outside 1..DDZ_PIMC_MAX_DETERMINIZATIONS,
 * B * D > INT_MAX or D * budget > INT_MAX: DDZ_E_ARG before any CUDA call.  The int32 sums cannot overflow when
 * D * budget * width <= 2^31 - 1. */
#define DDZ_PIMC_MAX_DETERMINIZATIONS 4096
int ddz_determinize(const void* state, const uint8_t* env_mask, int D, uint64_t seed, uint64_t env0, void* out_state,
                    int64_t* stats, int B, void* stream);
int ddz_uct_pool(const void* workspace, int budget, int D, int32_t* choice, uint64_t* move, int32_t* pooled_visits,
                 int32_t* pooled_wins, int B, void* stream);

/* Env.batch_arr2onehot over packed moves (envi.py:113,140-146): out float32[n][15][4] */
int ddz_encode_actions(const uint64_t* actions_u64, int64_t n, float* out, void* stream);

/* The Q-network's input for every legal move, built in place (net.py:81-90 repeats the face per action and torch.cat's the
 * action plane on): out float32 [n][C+1][15][4], row dst + i = [face of env b (C planes) | one-hot of move i of env b].
 * offsets / actions_u64: the lists of the CURRENT state (ddz_observe / ddz_rollout_step).  env_mask uint8[B] (or NULL):
 * only envs with a non-zero entry are written (e.g. the envs where the learning seat is to move); dst_offsets int32[B+1]
 * (or NULL = offsets): first output row of each env, e.g. the exclusive prefix sum of the selected envs' move counts. */
int ddz_encode_state_actions(const void* state, int variant, const int32_t* offsets, const uint64_t* actions_u64,
                             const uint8_t* env_mask, const int32_t* dst_offsets, float* out, int B, void* stream);

/* Batched DQNFirst.greedy_action / e_greedy_action (dqn.py:50-71): q float32[offsets[B]] are the Q-values the caller's
 * network gave to the legal moves (CSR order).  choice[b] = index of the first maximum of env b's segment, or of its first
 * NaN if it has one (torch.argmax semantics), or, with probability epsilon, a uniformly random index (Philox keyed by seed,
 * env0+b, stepno); -1 for an
 * env without legal moves (finished).  Feed choice to ddz_step / ddz_rollout_step with DDZ_CHOICE_INDEX. */
int ddz_select_actions(const float* q, const int32_t* offsets, float epsilon, uint64_t seed, uint64_t env0,
                       uint32_t stepno, int32_t* choice, int B, void* stream);

/* ---- host-buffer pipeline (the e2e path): one call per env-step does, without any Python in between,
 *   copy stream : H2D  host_choice (pinned, B x 4 bytes)  ->  dev_choice[k]            (k = step parity)
 *   main stream : wait; ddz_rollout_step(choice = dev_choice[k], DDZ_CHOICE_MOD, results -> results_dev)
 *   copy stream : wait; D2H  results_dev (first results_bytes of the contiguous r|done|cat|pad|reward block;
 *                       >= 3B, i.e. the reward floats are optional)  ->  results_host (pinned)
 * so the H2D of step t+1 and the D2H of step t-1 overlap the kernel of step t.  The pipe object only owns two CUDA
 * streams and a few events; every buffer stays caller-owned.  results_dev must alternate between two buffers (the
 * caller's ping-pong sets); results_host may rotate through up to DDZ_PIPE_DEPTH pinned buffers, so the host can read
 * the results of step t as late as while step t + DDZ_PIPE_DEPTH - 1 is being issued; ddz_pipe_wait(slot) blocks the
 * host until the D2H issued by the latest step with slot == step index % DDZ_PIPE_DEPTH has landed.  ddz_pipe_refill starts the upload of one slot of the deal pool into a
 * caller-provided staging buffer on a third copy stream and returns; the slot itself is replaced by a device-to-device
 * copy ordered between two steps, issued by the first ddz_pipe_step that finds the upload complete (so no step waits
 * for it), or by ddz_pipe_flush / the next ddz_pipe_refill, which do wait.  One upload can be in flight per pipe. */
#define DDZ_PIPE_DEPTH 4
typedef struct ddz_pipe ddz_pipe;
ddz_pipe* ddz_pipe_create(void);
void ddz_pipe_destroy(ddz_pipe* p);
int ddz_pipe_step(ddz_pipe* p, void* state, void* workspace, int variant,
                  const int32_t* prev_offsets, const uint64_t* prev_actions_u64,
                  const void* host_choice, void* dev_choice, uint64_t seed, uint64_t env0, uint32_t stepno,
                  const int32_t rewards[3], const int8_t* perm, const int8_t* lord_pile, int pool_games,
                  void* results_dev, void* results_host, size_t results_bytes,
                  int32_t* out_offsets, uint64_t* out_actions_u64, float* out_actions_f32, int64_t cap,
                  float* face, int64_t* stats, int B, void* stream);
int ddz_pipe_wait(ddz_pipe* p, int slot);
int ddz_pipe_refill(ddz_pipe* p, int8_t* pool_perm_slot, int8_t* pool_lord_slot, const int8_t* host_perm,
                    const int8_t* host_lord, int8_t* stage_perm, int8_t* stage_lord, int B, void* stream);
int ddz_pipe_flush(ddz_pipe* p, void* stream);   /* commit a staged deal-pool upload now (stream waits for it) */

/* ---- the same pipeline over several env groups of one GPU: ONE native call per env-step of all groups.
 * The envs of a GPU run as G independent groups (own state, workspace, ping-pong lists, stream) so that one group's
 * load-only prologue overlaps another group's store phase (DESIGN.md 4).  ddz_mpipe_step issues, for step s:
 *   copy stream   : H2D host_choice (pinned, sum(B_g) x 4 bytes, group-major) -> dev_choice
 *   stream g      : wait for it; ddz_rollout_step of group g (DDZ_CHOICE_MOD) with its slice of dev_choice; r | done | cat of
 *                   the group -> results_dev + 3 * off_g   (r[B_g] | done[B_g] | cat[B_g]; off_g = sum of B of the groups before g)
 *   copy stream 2 : wait for all groups' kernels; D2H results_dev (3 x sum(B_g) bytes) -> results_host (pinned)
 * The caller rotates dev_choice, results_dev and results_host through DDZ_PIPE_DEPTH buffers each (slot = step index %
 * DDZ_PIPE_DEPTH).  The step that reuses a slot first waits ON THE HOST (normally a no-op: the host reads results before
 * then) until the D2H of the step that used it before has landed, so no stream ever waits for an older step and the groups
 * never fall into lock-step.  4 G + 4 CUDA calls per step.  ddz_mpipe_wait(slot) blocks until the D2H of the latest step
 * with that slot has landed.  `gs` describes the groups FOR THIS STEP (prev_* = lists of the current state, out_* = the other
 * ping-pong set); reward (float32 [B_g][3], device) is optional and stays on the device.  stats may be one vector shared
 * by all groups (the kernels add atomically).  ddz_mpipe_refill starts the upload of one slot of every group's deal pool
 * from ONE pinned host array (rows group-major; it must stay valid until the slot is replaced) into a staging buffer on a
 * third copy stream.  The upload goes up in chunks of 384 KB, one with every following step, so that a step's entropy
 * never queues behind megabytes of permutations on the copy engine; each group's slot is replaced on the group's stream by
 * the first step that finds the upload complete, or by ddz_mpipe_flush / the next refill, which finish it and wait. */
#define DDZ_MPIPE_MAX_GROUPS 16
typedef struct {
    void* state; void* workspace;
    const int32_t* prev_offsets; const uint64_t* prev_actions_u64;
    int32_t* out_offsets; uint64_t* out_actions_u64; float* out_actions_f32; float* face;
    const int8_t* perm; const int8_t* lord_pile;   /* the group's deal pool [pool_games][B][54] / [pool_games][B] */
    float* reward;                                 /* device, optional */
    int64_t cap; uint64_t env0; int B; void* stream;
} ddz_group_step;
typedef struct ddz_mpipe ddz_mpipe;
ddz_mpipe* ddz_mpipe_create(int groups);
void ddz_mpipe_destroy(ddz_mpipe* p);
int ddz_mpipe_step(ddz_mpipe* p, const ddz_group_step* gs, int variant, const void* host_choice, void* dev_choice,
                   uint64_t seed, uint32_t stepno, const int32_t rewards[3], int pool_games,
                   void* results_dev, void* results_host, int64_t* stats);
int ddz_mpipe_wait(ddz_mpipe* p, int slot);
int ddz_mpipe_refill(ddz_mpipe* p, const ddz_group_step* gs, int8_t* const* pool_perm_slot, int8_t* const* pool_lord_slot,
                     const int8_t* host_perm, const int8_t* host_lord, int8_t* stage_perm, int8_t* stage_lord);
int ddz_mpipe_flush(ddz_mpipe* p, const ddz_group_step* gs);
/* make `stream` wait for the device-to-host copy of the latest step (e.g. to time a window with an event on that stream) */
int ddz_mpipe_join(ddz_mpipe* p, void* stream);

/* Optional allocator for the big float row buffers (actions_f32, face): device memory created compressible
 * (CU_MEM_ALLOCATION_COMP_GENERIC), so the L2 compresses the 0/1 thermometer rows on their way to HBM and expands them
 * for the reader -- transparent to every kernel, +15 % store bandwidth for this data.  The caller owns the buffer and
 * gives it back with ddz_rows_free(ptr, mapped_bytes); plain cudaMalloc / torch memory works everywhere as well.
 * Returns DDZ_E_CUDA (text in ddz_last_error) when the device or driver has no compressible memory. */
int ddz_rows_alloc(size_t bytes, int device, void** ptr, size_t* mapped_bytes);
int ddz_rows_free(void* ptr, size_t mapped_bytes);

/* env.face only (envi.py:87-217) */
int ddz_encode_face(const void* state, int variant, float* face, int B, void* stream);

/* Replay decode: the float transition rows a DQN minibatch needs (dqn.py:22-29 sample), rebuilt from packed states and moves.
 * A replay buffer that keeps each transition as two packed states (2 x 76 B) and two packed moves instead of float faces
 * and one-hot rows (2 x 240 (C + 1) B) decodes only the sampled rows, in one launch.
 * Sample i takes env rows[i] of `state` (a state of B envs) and its move moves[rows[i]] (uint64 [B]); rows are arbitrary,
 * duplicates and any order included.
 *   DDZ_ROWS_SPLIT:  face float32 [n][C][15][4] = what ddz_encode_face writes for that env, bit for bit; move_rows (optional)
 *                    float32 [n][15][4] = what ddz_encode_actions writes for that move (a pass, 0, is the zero row:
 *                    the reference's a1 = zeros of a terminal transition, game.py:123-124);
 *   DDZ_ROWS_CONCAT: face float32 [n][C+1][15][4], rows [face | move one-hot] = the Q-network input of net.py:88-90, the
 *                    rows ddz_encode_state_actions writes (move_rows must be NULL).
 * A row outside [0, B) gives all-zero rows and reads nothing.  n = 0 returns 0 without a launch.  NULL state / rows / face
 * with n > 0, n < 0, B <= 0, an unknown variant or layout, moves == NULL with DDZ_ROWS_CONCAT or with move_rows != NULL,
 * move_rows != NULL with DDZ_ROWS_CONCAT: DDZ_E_ARG before any CUDA call.  Form-B builds write the form-B rows. */
#define DDZ_ROWS_SPLIT 0
#define DDZ_ROWS_CONCAT 1
int ddz_encode_face_gather(const void* state, int variant, const int64_t* rows, int64_t n, const uint64_t* moves,
                           float* face, float* move_rows, int layout, int B, void* stream);

/* Action ids: a fixed index per move, the same in every position (the reference's action space, rule_based/utils/card.py:34-159,
 * which server/rule_utils/utils.py:21-38 get_mask_onehot60 masks).  The UNIVERSE is card.py's action_space in its order with
 * the 24 moves r.get_moves emits beyond it -- the {black joker, red joker} kicker pair of a two-trio 3+1 plane and of a 4+1+1
 * (server/mcts/get_moves.py:22-34) -- slotted in where card.py's combination loops would have produced them: 13 551 moves,
 * id 0 = pass.  (The card.py index of a move is its id minus the number of those 24 below it.)  Canonical legal lists are in
 * universe order, so the ids of a list strictly increase.  Ids do not depend on the probability form.
 *
 * ddz_move_ids: ids[i] = id of moves[i], -1 when moves[i] is not a move of the universe (counts no category produces, a
 * kicker equal to a main rank, a straight through '2', a nibble above 4, ...).
 * ddz_moves_of_ids: moves[i] = the packed move of ids[i]; an id outside [0, DDZ_NUM_ACTION_IDS) gives DDZ_MOVE_INVALID
 * (never a legal move: ddz_step with DDZ_CHOICE_MOVE treats it as an illegal choice).
 * n = 0 returns 0 without a launch; n < 0, or a NULL buffer with n > 0: DDZ_E_ARG before any CUDA call.
 *
 * ddz_legal_mask: one full row per env over the CURRENT lists (offsets / actions_u64 as ddz_observe, ddz_rollout_step or
 * ddz_legal_moves wrote them, holding cap moves):
 *   DDZ_MASK_BITS   out uint32 [B][DDZ_MASK_WORDS], bit (id & 31) of word (id >> 5); the 17 bits past id 13 550 are zero;
 *                   out 16-byte aligned;
 *   DDZ_MASK_BYTES  out uint8 [B][DDZ_NUM_ACTION_IDS], 1 for a legal id else 0 (a torch bool mask).
 * Every byte of every row is written.  Only list entries below cap are read: an env whose list runs past cap gets the stored
 * part and stats[7] (stats may be NULL) counts it once; a finished env (empty list) gets an all-zero row.
 * NULL offsets / out, actions_u64 NULL with cap > 0, cap < 0, B <= 0, an unknown layout or a misaligned bits row: DDZ_E_ARG
 * before any CUDA call. */
#define DDZ_NUM_ACTION_IDS 13551
#define DDZ_MOVE_INVALID 0xFFFFFFFFFFFFFFFFull
#define DDZ_MASK_BITS 0
#define DDZ_MASK_BYTES 1
#define DDZ_MASK_WORDS 424          /* ceil(DDZ_NUM_ACTION_IDS / 32) */
int ddz_move_ids(const uint64_t* moves, int64_t n, int32_t* ids, void* stream);
int ddz_moves_of_ids(const int32_t* ids, int64_t n, uint64_t* moves, void* stream);
int ddz_legal_mask(const int32_t* offsets, const uint64_t* actions_u64, int64_t cap, int layout, void* out, int64_t* stats,
                   int B, void* stream);

#ifdef __cplusplus
}
#endif
#endif
