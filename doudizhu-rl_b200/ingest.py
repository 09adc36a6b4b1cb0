"""Payload -> device state ingest (SURVEY.md 8f rank 3).

The reference's web bot rebuilds `face` / `valid_actions` from a JSON payload instead of a live env
(server/core.py:26-67, wire format server/client.py:6-24):

    {'role_id': 0|1|2,                      # 0 = up, 1 = lord, 2 = down: the player to move
     'cur_cards': [card values 3..17],      # its hand
     'history':    {0: [...], 1: [...], 2: [...]},   # everything each role has played
     'last_taken': {0: [...], 1: [...], 2: [...]},   # each role's most recent hand-out ([] = pass)
     'left':       {0: n0, 1: n1, 2: n2}}            # cards left per role

`env_from_payloads` packs a batch of such payloads into the state of a BatchedEnv*, after which `env.face` and
`env.valid_actions()` are produced by the same kernels as for a live game.  The other two players' hands are unknown:
only their SIZES enter the features (get_state_prob_manual, server/core.py:27), so they are filled with placeholder
cards of the right count.
"""
import numpy as np
import torch

from .env import BatchedEnvCooperationSimplify, pack_counts


def _counts(cards):
    c = np.zeros(15, np.int64)
    for v in cards:
        c[int(v) - 3] += 1
    return c


def _placeholder(n):
    """any hand with n cards (n <= 54): only its size is ever used"""
    c = np.zeros(15, np.int64)
    for r in range(15):
        take = min(4 if r < 13 else 1, n)
        c[r] = take
        n -= take
    if n:
        raise ValueError("a player cannot hold that many cards")
    return c


def payload_arrays(payloads):
    """list of payload dicts -> (role [B], hand [B,15], history [B,3,15], last_taken [B,3,15], left [B,3]) int64"""
    B = len(payloads)
    role = np.zeros(B, np.int64)
    hand = np.zeros((B, 15), np.int64)
    hist = np.zeros((B, 3, 15), np.int64)
    last = np.zeros((B, 3, 15), np.int64)
    left = np.zeros((B, 3), np.int64)
    for b, p in enumerate(payloads):
        role[b] = int(p["role_id"])
        hand[b] = _counts(p["cur_cards"])
        for q in range(3):
            hist[b, q] = _counts(p["history"][q] if q in p["history"] else p["history"][str(q)])
            last[b, q] = _counts(p["last_taken"][q] if q in p["last_taken"] else p["last_taken"][str(q)])
            left[b, q] = int(p["left"][q] if q in p["left"] else p["left"][str(q)])
    return role, hand, hist, last, left


def env_from_arrays(role, hand, hist, last, left, env_cls=BatchedEnvCooperationSimplify, hands=None, **kw):
    """hands (optional, int [B,3,15]): every role's real hand, for full-information positions such as the payload of the
    reference's MCTS bot (`hand_card`, server/mcts/interface.py:19-27); without it the other players get placeholders."""
    role, hand, hist, last, left = (np.asarray(x, np.int64) for x in (role, hand, hist, last, left))
    B = len(role)
    if ((role < 0) | (role > 2)).any() or (hand < 0).any() or (hand > 4).any() or (hist.sum(1) > 4).any():
        raise ValueError("bad payload: role_id must be 0..2 and no rank can appear more than four times")
    env = env_cls(B, **kw)
    if hands is not None:
        hands = np.asarray(hands, np.int64).reshape(B, 3, 15)
        if (hands[np.arange(B), role] != hand).any():
            raise ValueError("hands[b, role_id] must equal cur_cards")
    else:
        hands = np.zeros((B, 3, 15), np.int64)
        for b in range(B):
            for q in range(3):
                hands[b, q] = hand[b] if q == role[b] else _placeholder(int(left[b, q]))
    dev = env.device
    f, meta = env._fields()
    f[0:3] = pack_counts(torch.as_tensor(hands).to(dev)).t()
    f[3:6] = pack_counts(torch.as_tensor(hist).to(dev)).t()
    f[6:9] = pack_counts(torch.as_tensor(last).to(dev)).t()
    meta.copy_(torch.as_tensor(role, dtype=torch.int32).to(dev))      # role to move, not done, no deals consumed
    env._fresh = False
    return env


def env_from_payloads(payloads, env_cls=BatchedEnvCooperationSimplify, **kw):
    """BatchedEnv* whose env b is the position described by payloads[b] (server/core.py Predictor.face / valid_actions)"""
    return env_from_arrays(*payload_arrays(payloads), env_cls=env_cls, **kw)


def evaluate_moves(role, hands, hist, last, sims=256, seed=1, env_cls=None, device=None):
    """Flat Monte-Carlo evaluation of ONE full-information position (the job of the reference's MCTS bot,
    server/mcts/interface.py:15-45, with its random default policy but without the UCT tree): every legal move of the
    player to move is followed by `sims` random playouts to the end of the game (ddz_playout); returns
    (moves int64 [N,15], win_rate float [N]) where a win is a win of the mover's side."""
    from .env import BatchedEnv, unpack_counts
    env_cls = env_cls or BatchedEnv
    role = int(role)
    hands = np.asarray(hands, np.int64).reshape(3, 15)
    one = env_from_arrays([role], [hands[role]], [hist], [last], [hands.sum(1)], env_cls=env_cls, hands=[hands], device=device)
    moves = unpack_counts(one.actions_packed).cpu().numpy()
    n = len(moves)
    B = n * int(sims)
    env = env_from_arrays([role] * B, [hands[role]] * B, [hist] * B, [last] * B, [hands.sum(1)] * B, env_cls=env_cls,
                          hands=[hands] * B, seed=seed, device=device)
    first = torch.arange(n, device=env.device, dtype=torch.int32).repeat_interleave(int(sims))
    env.step(first)                       # env i plays move i // sims ...
    env.playout(max_steps=400)            # ... then everybody plays randomly to the end
    winner = env.winner.reshape(n, int(sims))
    mine = (winner == 1) if role == 1 else (winner != 1)
    return moves, mine.float().mean(1).cpu().numpy()


def mcts(payload, computation_budget=1000, seed=1, device=None, width=1, return_search=False, prune=True):
    """The entry point of the reference's search bot, `mcts(payload)` (server/mcts/interface.py:15-45), on the batched
    env: payload = {'role_id': 0|1|2, 'hand_card': {role: [card values 3..17]} for all three roles (full information),
    'last_taken': {role: [...]}}.  Returns the chosen move as a sorted list of card values ([] = pass).

    `computation_budget` iterations of the reference's UCT search (search.UctSearch: UCB selection, one expansion per
    iteration, random playout, back-up, answer = root child with the best win rate); the playouts run on the device,
    `width` of them per iteration (1 = the reference's sequential search); tree and playouts use the bot's pruned move
    lists (server/mcts/get_moves.py:36-69) unless prune=False.  evaluate_moves() above is the flat
    alternative: the same budget spread evenly over the root moves in ONE launch."""
    from .search import UctSearch
    role = int(payload["role_id"])
    get = lambda d, q: d[q] if q in d else d[str(q)]
    hands = np.stack([_counts(get(payload["hand_card"], q)) for q in range(3)])
    last = np.stack([_counts(get(payload["last_taken"], q)) for q in range(3)])
    search = UctSearch(role, hands, last, width=width, seed=seed, device=device, prune=prune)
    search.run(computation_budget)
    if not search.root.children:
        return ([], search) if return_search else []
    best = search.best_move()
    move = [r + 3 for r in range(15) for _ in range(int(best[r]))]
    return (move, search) if return_search else move


def mcts_batch(payloads, computation_budget=1000, seed=1, width=1, prune=True, device=None):
    """mcts(payload) for a whole list of payloads in ONE device launch (search.uct_search): the same full-information
    payloads ({'role_id', 'hand_card': {role: [...]} for all three roles, 'last_taken'}), one search tree per payload, all
    draws from Philox (so the answers are those of uct_search, not of the host-tree mcts()).  Returns one list of card
    values per payload ([] = pass, or no move to make)."""
    from .env import BatchedEnv
    from .search import uct_search
    get = lambda d, q: d[q] if q in d else d[str(q)]
    role = np.array([int(p["role_id"]) for p in payloads], np.int64)
    hands = np.stack([np.stack([_counts(get(p["hand_card"], q)) for q in range(3)]) for p in payloads])
    last = np.stack([np.stack([_counts(get(p["last_taken"], q)) for q in range(3)]) for p in payloads])
    B = len(payloads)
    env = env_from_arrays(role, hands[np.arange(B), role], np.zeros((B, 3, 15), np.int64), last, hands.sum(2),
                          env_cls=BatchedEnv, hands=hands, device=device)
    choice, moves = uct_search(env, computation_budget=computation_budget, width=width, prune=prune, seed=seed)
    out = []
    for ch, mv in zip(choice.tolist(), moves.tolist()):
        counts = [(mv >> (4 * r)) & 15 for r in range(15)] if ch >= 0 else [0] * 15
        out.append([r + 3 for r in range(15) for _ in range(counts[r])])
    return out


def unseen_mismatch(role, hand, hist, left):
    """indices of the positions whose unseen cards (full deck - own hand - everything played) cannot be the other two
    hands: a rank seen more often than the deck holds it, or an unseen count other than the sum of their `left` sizes"""
    role, hand, hist, left = (np.asarray(x, np.int64) for x in (role, hand, hist, left))
    deck = np.array([4] * 13 + [1, 1], np.int64)
    unseen = deck - hand - hist.sum(1)
    B = len(role)
    others = left[np.arange(B), (role + 1) % 3] + left[np.arange(B), (role + 2) % 3]
    return np.flatnonzero((unseen < 0).any(1) | (unseen.sum(1) != others))


def pimc_batch(payloads, determinizations=16, computation_budget=1000, seed=1, width=1, prune=True, device=None):
    """The search bot for a list of payloads in the web bot's wire format ({'role_id', 'cur_cards', 'history',
    'last_taken', 'left'}, server/client.py): the player sees only its own hand, so every payload is searched from that
    view (search.pimc_search: `determinizations` deals of the unseen cards, one UCT tree each, root statistics pooled).
    Returns one list of card values per payload ([] = pass), in the form mcts_batch uses.  Raises ValueError naming the
    payloads whose unseen cards do not match the other players' `left` counts."""
    from .env import BatchedEnv
    from .search import pimc_search
    role, hand, hist, last, left = payload_arrays(payloads)
    bad = unseen_mismatch(role, hand, hist, left)
    if len(bad):
        raise ValueError("payloads %s: the unseen cards do not match the other players' `left` counts" % bad.tolist())
    env = env_from_arrays(role, hand, hist, last, left, env_cls=BatchedEnv, device=device)
    choice, moves = pimc_search(env, determinizations=determinizations, computation_budget=computation_budget, width=width,
                                prune=prune, seed=seed)
    out = []
    for ch, mv in zip(choice.tolist(), moves.tolist()):
        counts = [(mv >> (4 * r)) & 15 for r in range(15)] if ch >= 0 else [0] * 15
        out.append([r + 3 for r in range(15) for _ in range(counts[r])])
    return out
