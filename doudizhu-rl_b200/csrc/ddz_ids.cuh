// ddz_ids.cuh -- action ids: a move's index in the fixed universe of 13 551 moves (the reference's action space, card.py:34-159,
// with the 24 rocket-kicker moves of r.get_moves where card.py's combination loops would have produced them), both ways, in
// closed form.  The universe is cut into blocks (make_action_ids.py): one main part with every k-subset of a kicker pool, in
// itertools.combinations order.  id = first id of the block + lexicographic rank of the kicker set (combinatorial number
// system over kBinom).  Canonical legal lists are in universe order, so their ids strictly increase.
#pragma once
#include "../../include/ddz_b200.h"
#include "ddz_device.cuh"

namespace ddz {

#include "ddz_action_ids.inc"

struct IdBlock { int first; uint32_t main, pool; int mult, kmult, k; };
DDZ_DEV IdBlock id_block(int i) {
    const uint64_t x = kIdBlocks[i];
    IdBlock o;
    o.first = (int)(x & 0xFFFFu); o.main = (uint32_t)(x >> 16) & 0x7FFFu; o.pool = (uint32_t)(x >> 32) & 0x7FFFu;
    o.mult = (int)(x >> 48) & 7; o.kmult = (int)(x >> 52) & 7; o.k = (int)(x >> 56) & 7;
    return o;
}

// a nibble above 4 (no rank has more than 4 cards), or anything above rank 14
DDZ_DEV bool bad_nibbles(uint64_t v) {
    const uint64_t m = 0x1111111111111111ull;
    const uint64_t b0 = v & m, b1 = (v >> 1) & m, b2 = (v >> 2) & m, b3 = (v >> 3) & m;
    return (v >> 60) != 0 || (b3 | (b2 & (b1 | b0))) != 0;
}

// lexicographic rank of the k-subset `set` of `pool` (the itertools.combinations order): C(n,k) - 1 - sum_i C(n-1-p_i, k-i),
// p_i = position in the pool of the i-th lowest element
DDZ_DEV int rank_combo(uint32_t set, uint32_t pool, int k) {
    const int n = __popc(pool);
    int r = binom(n, k) - 1;
    for (int i = 0; set; i++) {
        const uint32_t low = set & (0u - set);
        set ^= low;
        r -= binom(n - 1 - __popc(pool & (low - 1u)), k - i);
    }
    return r;
}

// id of a packed move, -1 if it is not a move.  classify() names the candidate block; the id's own move, rebuilt from that
// block and the kicker set, must equal the input (the round trip), so whatever classify guessed for a non-move gives -1.
DDZ_DEV int move_id(uint64_t mv) {
    if (mv == 0) return 0;
    if (bad_nibbles(mv)) return -1;
    const Trick t = classify(mv);
    int bi;
    if (t.cat <= 4 || t.cat == 12) {
        bi = kIdCatBlock[t.cat];
    } else if (t.cat <= 6 || t.cat >= 13) {
        if (t.val > 12) return -1;
        bi = kIdCatBlock[t.cat] + t.val;
    } else {                                               // lines: blocks by start, then by length
        const int c = t.cat - 7;
        if (t.val > 11 || t.len < kIdLineMin[c] || t.len > kIdLineMax[c] || t.val + t.len > 12) return -1;
        bi = kIdLineBlock[c][t.val] + t.len - kIdLineMin[c];
    }
    const IdBlock blk = id_block(bi);
    const uint32_t kick = masks_of(mv).g1 & ~blk.main;
    if (__popc(kick) != blk.k || (kick & ~blk.pool) != 0) return -1;
    if (pack_move(blk.main, blk.mult, kick, blk.kmult) != mv) return -1;
    return blk.first + rank_combo(kick, blk.pool, blk.k);
}

// packed move of an id, DDZ_MOVE_INVALID outside [0, DDZ_NUM_ACTION_IDS)
DDZ_DEV uint64_t move_of_id(int id) {
    if (id < 0 || id >= DDZ_NUM_ACTION_IDS) return DDZ_MOVE_INVALID;
    int lo = 0, hi = DDZ_ID_BLOCKS - 1;                    // the last block whose first id is <= id
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((int)(kIdBlocks[mid] & 0xFFFFu) <= id) lo = mid; else hi = mid - 1;
    }
    const IdBlock blk = id_block(lo);
    return pack_move(blk.main, blk.mult, unrank_combo(blk.pool, blk.k, id - blk.first), blk.kmult);
}

}  // namespace ddz
