"""The determinized search (ddz_determinize -> ddz_uct_search over B * D roots -> ddz_uct_pool, search.pimc_search)
restated on the CPU from the draw and pooling rules of include/ddz_b200.h, with no product code:
  * determinize: the unseen cards (deck - mover's hand - hist[0..2]) walked in rank order, card j going to role
    a = (m+1)%3 when philox(seed, (env0 + b) * D + d, 0xC0000000 + j) % (ra + rc) < ra, else to c = (m+2)%3;
  * the D trees of a root searched by the C port over the oracle (uct_philox_reference.ref_uct_batch, env0 * D);
  * pool: root children's visits and wins added up per canonical index, answer = best pooled wins / visits with exact
    integer comparison, lowest index on ties.
philox_np is Philox4x32-10 over numpy arrays, equal to oracle.philox (asserted in test_pimc.py).
TEST INFRASTRUCTURE ONLY."""
import numpy as np

from uct_philox_reference import ref_uct_batch

DET_STEP = 0xC0000000
DECK = np.array([4] * 13 + [1, 1], np.int64)
MAX_LEGAL = 512
M32 = np.uint64(0xFFFFFFFF)


def philox_np(seed, env, step):
    """philox(seed, env, step) (oracle.philox, ddz_device.cuh) for arrays of env / step: uint32 array"""
    env = np.asarray(env, np.uint64)
    step = np.asarray(step, np.uint64)
    env, step = np.broadcast_arrays(env, step)
    c0, c1 = env & M32, env >> np.uint64(32)
    c2, c3 = step & M32, np.zeros_like(env)
    k0, k1 = np.uint64(int(seed) & 0xFFFFFFFF), np.uint64((int(seed) >> 32) & 0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        h0, l0 = p0 >> np.uint64(32), p0 & M32
        h1, l1 = p1 >> np.uint64(32), p1 & M32
        c0, c1, c2, c3 = h1 ^ c1 ^ k0, l1, h0 ^ c3 ^ k1, l0
        k0 = (k0 + np.uint64(0x9E3779B9)) & M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & M32
    return c0.astype(np.uint32)


def determinize(hands, hist, recent, meta, D, seed, env0=0, mask=None):
    """hands / hist / recent int [B,3,15], meta uint32 [B] -> (hands, hist, recent, meta) of the B * D output envs (env
    b * D + d = determinization d of env b) and the number of inconsistent roots (stats[7])"""
    hands, hist, recent = (np.asarray(x, np.int64) for x in (hands, hist, recent))
    meta = np.asarray(meta, np.uint32)
    B = len(meta)
    live = ((meta >> 2) & 1) == 0
    if mask is not None:
        live &= np.asarray(mask, bool)
    m = (meta & 3).astype(np.int64)
    a, c = (m + 1) % 3, (m + 2) % 3
    ar = np.arange(B)
    unseen = DECK[None, :] - hands[ar, m] - hist.sum(1)
    na, nc = hands[ar, a].sum(1), hands[ar, c].sum(1)
    bad = live & ((unseen < 0).any(1) | (unseen.sum(1) != na + nc))
    good = live & ~bad
    out_h = np.repeat(hands, D, axis=0)
    out_meta = np.repeat(meta, D).copy()
    out_meta[np.repeat(bad, D)] |= np.uint32(4 | 32)
    rows = np.flatnonzero(np.repeat(good, D))
    if len(rows):
        b = rows // D
        d = rows % D
        ctr = ((np.uint64(env0) + b.astype(np.uint64)) * np.uint64(D) + d.astype(np.uint64))
        U = unseen[b].sum(1)
        cards = np.full((len(rows), 54), -1, np.int64)        # the unseen cards of each row in rank order
        for i, row in enumerate(unseen[b]):
            cs = np.repeat(np.arange(15), row)
            cards[i, :len(cs)] = cs
        ra, rc = na[b].copy(), nc[b].copy()
        ha = np.zeros((len(rows), 15), np.int64)
        hc = np.zeros((len(rows), 15), np.int64)
        for j in range(int(U.max()) if len(U) else 0):
            on = j < U
            u = philox_np(seed, ctr, DET_STEP + j).astype(np.int64)
            tot = np.maximum(ra + rc, 1)
            to_a = on & ((u % tot) < ra)
            to_c = on & ~to_a
            idx = np.flatnonzero(to_a)
            np.add.at(ha, (idx, cards[idx, j]), 1)
            idx = np.flatnonzero(to_c)
            np.add.at(hc, (idx, cards[idx, j]), 1)
            ra -= to_a
            rc -= to_c
        assert (ra == 0).all() and (rc == 0).all()
        out_h[rows, a[b]] = ha
        out_h[rows, c[b]] = hc
    return out_h, np.repeat(hist, D, axis=0), np.repeat(recent, D, axis=0), out_meta, int(bad.sum())


def better(w1, v1, w2, v2):
    """wins / visits w1 / v1 strictly above w2 / v2 (exact)"""
    return int(w1) * int(v2) > int(w2) * int(v1)


def pool(trees, D):
    """ddz_uct_pool over the arrays of ref_uct_batch (parent, visits, wins, index [B*D, n], nnodes [B*D]):
    (choice int32 [B], pooled_visits int64 [B,512], pooled_wins int64 [B,512])"""
    nnodes = np.asarray(trees["nnodes"])
    B = len(nnodes) // D
    pv = np.zeros((B, MAX_LEGAL), np.int64)
    pw = np.zeros((B, MAX_LEGAL), np.int64)
    choice = np.full(B, -1, np.int32)
    for b in range(B):
        searched = False
        for t in range(b * D, b * D + D):
            n = int(nnodes[t])
            if n <= 0:
                continue
            searched = True
            for k in range(1, n):
                if trees["parent"][t][k] == 0:
                    pv[b, trees["index"][t][k]] += int(trees["visits"][t][k])
                    pw[b, trees["index"][t][k]] += int(trees["wins"][t][k])
        if not searched:
            continue
        best = -1
        for k in np.flatnonzero(pv[b] > 0):
            if best < 0 or better(pw[b, k], pv[b, k], pw[b, best], pv[b, best]):
                best = int(k)
        choice[b] = best
    return choice, pv, pw


def pimc_reference(oracle, hands, hist, recent, meta, D, budget, width=1, prune=True, c=0.7, seed=1, env0=0, mask=None):
    """determinize -> ref_uct_batch(env0 = env0 * D) -> pool: dict choice [B], move uint64 [B] (~0: none),
    pooled_visits / pooled_wins [B,512], and the determinized hands and meta"""
    h, _, r, mt, nbad = determinize(hands, hist, recent, meta, D, seed, env0=env0, mask=mask)
    live = ((mt >> 2) & 1) == 0
    if mask is not None:
        live &= np.repeat(np.asarray(mask, bool), D)
    trees = ref_uct_batch(h, r, (mt & 3).astype(np.int32), live, budget, width=width, prune=prune, c=c, seed=seed,
                          env0=env0 * D)
    choice, pv, pw = pool(trees, D)
    move = np.full(len(choice), np.uint64(2 ** 64 - 1), np.uint64)
    for b, k in enumerate(choice):
        if k >= 0:
            m = int(mt[b * D] & 3)
            rec = np.asarray(recent[b], np.int64)
            last = rec[(m + 2) % 3] if rec[(m + 2) % 3].any() else rec[(m + 1) % 3]
            move[b] = np.uint64(oracle.pack(oracle.get_moves(np.asarray(hands[b][m]), last, fast=True)[k]))
    return {"choice": choice, "move": move, "pooled_visits": pv, "pooled_wins": pw, "hands": h, "meta": mt,
            "errors": nbad, "trees": trees}
