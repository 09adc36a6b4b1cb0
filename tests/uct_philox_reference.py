"""The reference's UCT search (tests/uct_reference_algorithm.py::uct, server/mcts/interface.py:37-45) with the draw rule of
the batched device search (ddz_uct_search, include/ddz_b200.h): every random draw comes from Philox, so the Python
restatement, the C port over the oracle (host_harness/uct_oracle.c, `ref_uct_batch` below) and the kernel can agree bit
for bit.
  * tree draw j of root b:  philox(seed, env0 + b, 0x80000000 + j) -- the expansion draw (u % remaining, also with one
    entry left) and the tie draw among k >= 2 exactly equal values (u % k), in the order they happen;
  * playout w of iteration it:  philox(seed, ((env0 + b) * budget + it) * width + w, t) at its decision t.
TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import math
import os
import subprocess

import numpy as np

from uct_reference_algorithm import Node, State, pruned_playout_step

TREE_STEP = 0x80000000
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "host_harness", "uct_oracle.c")
ORACLE_SRC = [os.path.join(ROOT, "oracle", f) for f in ("ddz_oracle.c", "ddz_oracle.h")]
LIB = os.path.join(HERE, "host_harness", "libuct_oracle.so")


def uct(oracle, role, hands, recent, budget, width=1, c=0.7, seed=1, prune=True, env=0):
    """returns (best move int64[15] or None, nodes in creation order); env = env0 + b of the root"""
    me = int(role)
    draws = [0]
    root = Node(None, State(np.asarray(hands, np.int64).copy(), np.asarray(recent, np.int64).copy(), me, -1, None))
    root.index, nodes = -1, [root]

    def draw():
        u = oracle.philox(seed, env, TREE_STEP + draws[0])
        draws[0] += 1
        return u

    def won(winner):
        return 1 if (winner == 1) == (me == 1) else 0

    def pick(values, target):                                          # a random one among exact ties
        tied = np.flatnonzero(values == target)
        return int(tied[0] if len(tied) == 1 else tied[draw() % len(tied)])

    def entries(st):
        last = st.last_move()
        lst = oracle.mcts_moves(st.hands[st.player], last) if prune else oracle.get_moves(st.hands[st.player], last, fast=True)
        return [m.astype(np.int64) for m in lst]

    def tree_policy(node):
        while node.state.winner == -1:
            if node.untried is None:
                node.untried = entries(node.state)
                node.nmoves = len(node.untried)
            if len(node.children) < node.nmoves:                       # list.pop(i) of the i-th remaining entry
                mv = node.untried.pop(draw() % len(node.untried))
                st = node.state
                full = oracle.get_moves(st.hands[st.player], st.last_move(), fast=True).astype(np.int64)
                sub = Node(node, st.play(mv))
                sub.index = int(np.flatnonzero((full == mv).all(axis=1))[0])
                node.children.append(sub)
                nodes.append(sub)
                return sub
            visit = np.array([n.visit for n in node.children], np.float64)
            reward = np.array([n.reward for n in node.children], np.float64)
            values = reward / visit + c * np.sqrt(2.0 * math.log(node.visit) / visit)
            node = node.children[pick(values, values.max() if node.state.player == me else values.min())]
        return node

    def default_policy(node, it):
        st = node.state
        if st.winner != -1:
            return width * won(st.winner)
        rb = oracle.RefBatch(width, 0)
        rb.envs["hand"][:] = st.hands
        rb.envs["recent"][:] = st.recent
        rb.envs["cur"] = st.player
        rb.envs["winner"] = -1
        env0 = (env * budget + it) * width                            # playout w draws from stream env0 + w
        t = 0
        while not rb.envs["done"].all():
            if prune:
                pruned_playout_step(oracle, rb, seed, env0, t)
            else:
                rb.observe(want_f32=False, want_face=False)
                rb.step(mode=2, seed=seed, env0=env0, step=t)
            t += 1
        return sum(won(int(w)) for w in rb.envs["winner"])

    if root.state.winner == -1 and not entries(root.state):
        return None, []
    for it in range(budget):
        node = tree_policy(root)
        reward = default_policy(node, it)
        while node is not None:
            node.visit += width
            node.reward += reward
            node = node.parent
    rate = np.array([n.reward / n.visit for n in root.children])
    best = root.children[pick(rate, rate.max())]
    return best.state.action, nodes


def lib():
    deps = [SRC] + ORACLE_SRC
    if not os.path.exists(LIB) or any(os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-pthread", "-fno-fast-math",
                               "-ffp-contract=off", "-o", LIB, SRC, ORACLE_SRC[0], "-lm"])
    L = C.CDLL(LIB)
    vp = C.c_void_p
    L.ddz_ref_uct_batch.argtypes = [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_uint64, C.c_uint64,
                                    C.c_int] + [vp] * 9
    return L


def ref_uct_batch(hands, recent, cur, live, budget, width=1, prune=True, c=0.7, seed=1, env0=0, nthreads=None):
    """ddz_ref_uct_batch over B roots (hands / recent int [B,3,15], cur int [B], live bool [B]): dict of numpy arrays
    choice, move, root_n, nnodes [B] and parent, visits, wins, index, node_move [B, budget + 1] (creation order)"""
    hands = np.ascontiguousarray(hands, np.int8)
    recent = np.ascontiguousarray(recent, np.int8)
    cur = np.ascontiguousarray(cur, np.int32)
    live = np.ascontiguousarray(live, np.uint8)
    B = len(cur)
    out = {k: np.zeros(B, np.int32) for k in ("choice", "root_n", "nnodes")}
    out["move"] = np.zeros(B, np.uint64)
    for k in ("parent", "visits", "wins", "index"):
        out[k] = np.zeros((B, budget + 1), np.int32)
    out["node_move"] = np.zeros((B, budget + 1), np.uint64)
    p = lambda a: a.ctypes.data
    rc = lib().ddz_ref_uct_batch(p(hands), p(recent), p(cur), p(live), B, int(budget), int(width), int(prune), float(c),
                                 int(seed), int(env0), int(nthreads or os.cpu_count() or 1), p(out["choice"]),
                                 p(out["move"]), p(out["root_n"]), p(out["nnodes"]), p(out["parent"]), p(out["visits"]),
                                 p(out["wins"]), p(out["index"]), p(out["node_move"]))
    assert rc == 0
    return out
