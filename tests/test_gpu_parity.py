"""GPU parity: the CUDA path, called through the C-ABI (ddz_b200 -> ctypes -> libddz_b200.so), against the CPU oracle
and the committed golden fixtures.  Everything is integer / exact-float work: comparisons are bit-exact."""
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


def _rand_hands(rng, n, lo=1, hi=21):
    deck = np.array([i // 4 for i in range(52)] + [13, 14])
    return np.stack([np.bincount(rng.permutation(deck)[:rng.integers(lo, hi)], minlength=15) for _ in range(n)]).astype(np.int8)


def _split(packed, offsets):
    packed = packed.cpu().numpy().view(np.uint64)
    off = offsets.cpu().numpy()
    return [packed[off[i]:off[i + 1]] for i in range(len(off) - 1)]


# ------------------------------------------------------------------ legal moves (r.get_moves)
def test_get_moves_golden_legal_sets(D, oracle, golden):
    g = golden.legal_sets
    packed, offsets = D.get_moves(g["hands"], g["lasts"])
    lists = _split(packed, offsets)
    off = g["legal_off"]
    for i, got in enumerate(lists):
        want = oracle.pack(g["universe"][g["legal_idx"][off[i]:off[i + 1]]])
        assert np.array_equal(got, want), (i, g["hands"][i], g["lasts"][i])


def test_get_moves_random_vs_oracle(D, oracle):
    rng = np.random.default_rng(11)
    n = 6000
    hands = _rand_hands(rng, n)
    z = np.zeros(15, np.int8)
    lasts = np.zeros((n, 15), np.int8)
    for i in range(n):
        if i % 3:
            om = oracle.get_moves(_rand_hands(rng, 1, 2, 21)[0], z, fast=True)
            w = om.sum(1).astype(np.float64) ** 2
            lasts[i] = om[rng.choice(len(om), p=w / w.sum())]
    packed, offsets = D.get_moves(hands, lasts)
    for i, got in enumerate(_split(packed, offsets)):
        want = oracle.pack(oracle.get_moves(hands[i], lasts[i], fast=(i % 7 != 0)))
        assert np.array_equal(got, np.atleast_1d(want)), (i, hands[i], lasts[i])


def test_get_moves_adversarial_and_edges(D, oracle):
    z = np.zeros(15, np.int8)
    worst = np.array([1, 3, 3, 3, 3, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0], np.int8)
    hands = np.stack([worst, z, z, np.array([4] * 5 + [0] * 10, np.int8),
                      np.array([3, 3, 3, 3, 3, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0], np.int8)])
    single = np.eye(15, dtype=np.int8)[3]
    lasts = np.stack([z, z, single, z, z])
    packed, offsets = D.get_moves(hands, lasts)
    lists = _split(packed, offsets)
    assert len(lists[0]) == 497 and len(lists[1]) == 0 and list(lists[2]) == [0]
    for i in range(len(hands)):
        assert np.array_equal(lists[i], np.atleast_1d(oracle.pack(oracle.get_moves(hands[i], lasts[i]))))


def test_encode_actions_kernel(D, oracle):
    cnt = oracle.universe()[0]
    packed = torch.as_tensor(oracle.pack(cnt).view(np.int64)).cuda()
    out = D.BatchedEnv.encode_actions(packed).cpu().numpy()
    want = (np.arange(4)[None, None, :] < cnt[:, :, None]).astype(np.float32)
    assert np.array_equal(out, want)


# ------------------------------------------------------------------ full rollouts
def _compare_observation(env, ref, t, check_f32=True):
    B = env.B
    off, au, af, face = ref.observe(want_f32=check_f32)
    assert np.array_equal(env.offsets.cpu().numpy(), off), "offsets, step %d" % t
    assert np.array_equal(env.actions_packed.cpu().numpy().view(np.uint64), au), "legal lists, step %d" % t
    if check_f32:
        assert np.array_equal(env.valid_actions()[0].cpu().numpy(), af), "action one-hots, step %d" % t
    assert np.array_equal(env.face.cpu().numpy(), face), "face, step %d" % t
    return int(off[B])


def _compare_state(env, ref, t):
    f, meta = ref.export()
    ef, emeta = env._fields()
    assert np.array_equal(ef.cpu().numpy().view(np.uint64), f), "state fields, step %d" % t
    assert np.array_equal(emeta.cpu().numpy().view(np.uint32), meta), "meta, step %d" % t


@pytest.mark.parametrize("cls,variant", [("BatchedEnv", 0), ("BatchedEnvComplicated", 1),
                                         ("BatchedEnvCooperation", 2), ("BatchedEnvCooperationSimplify", 3)])
def test_fused_rollout_bit_exact(D, oracle, cls, variant):
    """BASELINE config 2: 4096 envs, random play from the Philox index stream, >= 3 games per env; every legal list,
    encoded tensor, return value and the full state compared with the oracle at every step."""
    B, G, seed = 4096, 8, 20260101
    steps = 220 if variant == 2 else 60
    perm, lord = D.random_deals(B, seed=5, pool_games=G)
    perm_d, lord_d = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = getattr(D, cls)(B, seed=seed, env0=1000)
    env.prepare(perm_d, lord_d, pool_games=G)
    ref = oracle.RefBatch(B, variant)
    ref.deal(perm, lord, pool_games=G)
    env.observe()
    for t in range(steps):
        _compare_observation(env, ref, t, check_f32=(t % 8 == 0))
        r, done, cat = env.rollout_step(mode=D.native.CHOICE_PHILOX, perm=perm_d, lord_pile=lord_d, pool_games=G)
        rr, rd, rc, rrew = ref.step(mode=2, seed=seed, env0=1000, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=G)
        assert np.array_equal(r.cpu().numpy(), rr) and np.array_equal(done.cpu().numpy(), rd)
        assert np.array_equal(cat.cpu().numpy(), rc) and np.array_equal(env.reward.cpu().numpy(), rrew)
        if t % 16 == 0:
            _compare_state(env, ref, t)
    _compare_state(env, ref, steps)
    stats = env.stats.cpu().numpy()
    assert np.array_equal(stats[[0, 1, 2, 3, 4, 5, 6, 9]], ref.stats[[0, 1, 2, 3, 4, 5, 6, 9]])
    assert stats[7] == 0
    if variant == 2:
        assert stats[0] >= 3 * B * 0.8                      # about 62 decisions per game
        assert stats[1] + stats[2] + stats[3] == stats[0]


def test_unfused_api_matches_oracle(D, oracle):
    """reset / prepare / observe / step (index), step_random (host entropy), step_manual (one-hot) one by one."""
    B = 512
    rng = np.random.default_rng(3)
    perm, lord = D.random_deals(B, seed=8)
    env = D.BatchedEnvCooperation(B, debug=True)
    env.prepare(perm, lord)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord)
    for t in range(90):
        n = _compare_observation(env, ref, t)
        off = ref.offsets
        cnt = np.diff(off)
        kind = t % 3
        if kind == 0:
            choice = np.where(cnt > 0, rng.integers(0, 1 << 30, B) % np.maximum(cnt, 1), 0).astype(np.int32)
            r, done, cat = env.step(choice)
            rr, rd, rc, rrew = ref.step(choice, mode=0)
        elif kind == 1:
            ent = rng.integers(0, 1 << 32, B, dtype=np.uint64).astype(np.uint32)
            r, done, cat = env.step_random(ent)
            rr, rd, rc, rrew = ref.step(ent.view(np.int32), mode=1)
        else:
            choice = np.where(cnt > 0, rng.integers(0, 1 << 30, B) % np.maximum(cnt, 1), 0).astype(np.int32)
            acts, offs = env.valid_actions()
            idx = torch.as_tensor(off[:-1].astype(np.int64) + choice).cuda()
            idx = torch.where(torch.as_tensor(cnt > 0).cuda(), idx, torch.zeros_like(idx))
            onehot = acts[idx]
            # finished envs have no list: give them an all-zero one-hot (ignored)
            onehot = onehot * torch.as_tensor(cnt > 0).cuda()[:, None, None]
            r, done, cat = env.step_manual(onehot)
            rr, rd, rc, rrew = ref.step(choice, mode=0)
        assert np.array_equal(r.cpu().numpy(), rr) and np.array_equal(done.cpu().numpy(), rd), t
        assert np.array_equal(cat.cpu().numpy(), rc) and np.array_equal(env.reward.cpu().numpy(), rrew), t
        _compare_state(env, ref, t)
        # getters
        if t % 10 == 0:
            f, meta = ref.export()
            assert np.array_equal(env.left.cpu().numpy(), oracle.unpack(f[0:3].T).sum(-1))
            assert np.array_equal(env.history.cpu().numpy(), oracle.unpack(f[3:6].T))
            assert np.array_equal(env.recent_handout.cpu().numpy(), oracle.unpack(f[6:9].T))
            assert np.array_equal(env.get_role_ID().cpu().numpy(), (meta & 3) + 1)
        if t == 70:   # re-deal the finished ones, keep the others
            perm2, lord2 = D.random_deals(B, seed=9)
            env.prepare(perm2, lord2, only_done=True)
            ref.deal(perm2, lord2, only_done=True)


def test_reference_api_views_replay_golden_trace(D, golden):
    """The B=1 `Env*` views expose the reference's exact signatures; replay the golden envi.py trace through them."""
    t = golden.envi_trace
    classes = [(D.Env, "face_first"), (D.EnvComplicated, "face_complicated"),
               (D.EnvCooperation, "face_cooperation"), (D.EnvCooperationSimplify, "face_simplify")]
    for cls, key in classes:
        faces = t[key]
        env = cls(debug=True)
        fi = li = 0
        for g in range(4):
            env.reset()
            env.prepare(t["perms"][g][None], np.zeros(1, np.int8))
            for s in np.flatnonzero(t["game"] == g):
                n = int(t["n_legal"][s])
                face = env.face
                assert tuple(face.shape) == faces[fi].shape and face.dtype == torch.float32
                assert np.array_equal(face.cpu().numpy(), faces[fi])
                acts = env.valid_actions()
                assert tuple(acts.shape) == (n, 15, 4)
                assert np.array_equal(acts.cpu().numpy(), t["actions_f32"][li:li + n])
                assert env.valid_actions(tensor=False) == t["legal"][li:li + n].tolist()
                assert env.get_role_ID() - 1 == t["role"][s]
                r, done, cat = env.step_manual(acts[int(t["choice"][s])])
                assert (r, done, cat) == (int(t["r"][s]), bool(t["done"][s]), int(t["cat"][s]))
                assert np.array_equal(env.left, t["left"][s]) and np.array_equal(env.taken, t["taken"][s])
                for q in range(3):
                    assert np.array_equal(env.history[q], t["history"][s][q])
                    assert np.array_equal(env.recent_handout[q], t["recent"][s][q])
                fi += 1
                li += n
            assert np.array_equal(env.face.cpu().numpy(), faces[fi])      # terminal face (game.py:121-122)
            fi += 1


def test_encode_face_standalone(D, oracle):
    B = 300
    perm, lord = D.random_deals(B, seed=21)
    for variant, cls in enumerate([D.BatchedEnv, D.BatchedEnvComplicated, D.BatchedEnvCooperation, D.BatchedEnvCooperationSimplify]):
        env = cls(B)
        env.prepare(perm, lord)
        ref = oracle.RefBatch(B, variant)
        ref.deal(perm, lord)
        for t in range(5):
            env.rollout_step()
            off, au, af, face = ref.observe()
            ref.step(mode=2, seed=0, env0=0, step=t)
        out = torch.empty_like(env._face)
        D.native.check(D.native.lib.ddz_encode_face(env._state.data_ptr(), variant, out.data_ptr(), B, None), "ddz_encode_face")
        torch.cuda.synchronize()
        _, _, _, face = ref.observe()
        assert np.array_equal(out.cpu().numpy(), face)


def test_errors_are_flagged_not_silent(D):
    B = 64
    perm, lord = D.random_deals(B, seed=2)
    env = D.BatchedEnv(B)
    env.prepare(perm, lord)
    before = env._state.clone()
    bad = torch.full((B,), 10_000, dtype=torch.int32)
    r, done, cat = env.step(bad)
    torch.cuda.synchronize()
    assert int(env.stats[7].item()) == B and (cat == -1).all() and (r == 0).all()
    f0 = before[: 18 * B]
    assert torch.equal(env._state[: 18 * B], f0)                       # cards untouched
    assert ((env._fields()[1] >> 5) & 1).all()                         # sticky error bit
    # a bad permutation is refused
    env2 = D.BatchedEnv(B, debug=True)
    badperm = perm.copy()
    badperm[5, 0] = badperm[5, 1]
    with pytest.raises(D.native.DdzError):
        env2.prepare(badperm, lord)
    # too small an action buffer is reported (stats[7]); asking for the lists then grows it and observes again
    env3 = D.BatchedEnv(B, max_actions_per_env=4)
    env3.prepare(perm, lord)
    env3.observe()
    torch.cuda.synchronize()
    assert int(env3.stats[7].item()) == 1 and int(env3._offsets[env3._cur][B].item()) > env3.cap == 4 * B
    n = env3.num_actions
    assert env3.cap >= n > 4 * B and int(env3.offsets[B].item()) == n and int(env3.stats[7].item()) == 1
    # null / bad arguments come back as error codes, not crashes
    assert D.native.lib.ddz_observe(None, None, 0, None, None, None, 0, None, None, B, None) == D.native.E_ARG
    assert D.native.lib.ddz_reset(None, None, None, 1, 0, None, B, None) == D.native.E_ARG
    assert D.native.lib.ddz_face_channels(7) == D.native.E_ARG


def test_state_dict_resume_is_exact(D):
    B = 256
    perm, lord = D.random_deals(B, seed=4, pool_games=2)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    a = D.BatchedEnvCooperation(B, seed=77)
    a.prepare(pd, ld, pool_games=2)
    for _ in range(30):
        a.rollout_step(perm=pd, lord_pile=ld, pool_games=2)
    sd = a.state_dict()
    b = D.BatchedEnvCooperation(B, seed=77)
    b.load_state_dict(sd)
    for _ in range(40):
        a.rollout_step(perm=pd, lord_pile=ld, pool_games=2)
        b.rollout_step(perm=pd, lord_pile=ld, pool_games=2)
    keep = [0, 1, 2, 3, 4, 5, 6, 7, 9]        # stats[8] (moves emitted) also counts b's extra observe() after the load
    assert torch.equal(a._state, b._state) and torch.equal(a.face, b.face) and torch.equal(a.stats[keep], b.stats[keep])
    assert torch.equal(a.offsets, b.offsets) and torch.equal(a.actions_packed, b.actions_packed)


def test_cuda_graph_replay_matches_oracle(D, oracle):
    """GraphedRollout: the captured ping-pong pair, replayed with the device-side step counter, follows the same
    Philox stream as explicit stepping."""
    B, G, seed = 1024, 4, 99
    perm, lord = D.random_deals(B, seed=12, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, seed=seed)
    env.prepare(pd, ld, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    t = 0
    for _ in range(3):                       # a few explicit steps first: the counter must carry over
        ref.observe(want_f32=False, want_face=False)
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
        ref.step(mode=2, seed=seed, step=t); ref.deal(perm, lord, only_done=True, pool_games=G); t += 1
    gr = D.GraphedRollout(env, pd, ld, G)
    for _ in range(40):
        gr.replay()
        for _ in range(2):
            ref.observe(want_f32=False, want_face=False)
            ref.step(mode=2, seed=seed, step=t); ref.deal(perm, lord, only_done=True, pool_games=G); t += 1
    _compare_observation(env, ref, t)
    _compare_state(env, ref, t)
    env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)     # and explicit stepping continues seamlessly
    ref.step(mode=2, seed=seed, step=t); ref.deal(perm, lord, only_done=True, pool_games=G)
    _compare_observation(env, ref, t + 1)
    assert int(env.stats[7].item()) == 0


def test_host_rollout_pipeline_matches_oracle(D, oracle):
    """HostRollout: entropy from pinned host memory every step, deal-pool slots refilled from the host, results read
    back into pinned memory -- with the copies on their own streams.  Every step's results must equal the oracle's."""
    B, G = 2048, 2
    rng = np.random.default_rng(31)
    perm, lord = D.random_deals(B, seed=13, pool_games=G)
    pool = [np.array(perm.reshape(G, B, 54)), np.array(lord.reshape(G, B))]
    env = D.BatchedEnvCooperation(B)
    env.prepare(perm, lord, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    host = D.HostRollout(env, perm, lord, G, fetch_reward=True)
    ents = [torch.as_tensor(rng.integers(0, 1 << 31, B).astype(np.int32)).pin_memory() for _ in range(6)]
    pending = []
    for t in range(120):
        if t % 40 == 20:                              # refresh slot (t // 40) % G with new host-made deals
            slot = (t // 40) % G
            p2, l2 = D.random_deals(B, seed=100 + t)
            host.refill(slot, torch.as_tensor(p2).pin_memory(), torch.as_tensor(l2).pin_memory(), now=True)
            pool[0][slot], pool[1][slot] = p2, l2
        res = host.step(ents[t % 6])
        ref.observe(want_f32=False, want_face=False)
        want = ref.step(ents[t % 6].numpy(), mode=1)
        ref.deal(pool[0].reshape(-1, 54), pool[1].reshape(-1), only_done=True, pool_games=G)
        pending.append((res, [w.copy() for w in want]))
        if len(pending) == 2:                         # results of step t-1 are read while step t is in flight
            got, (rr, rd, rc, rrew) = pending.pop(0)
            D.HostRollout.wait(got)
            assert np.array_equal(got.r.numpy(), rr) and np.array_equal(got.done.numpy(), rd), t
            assert np.array_equal(got.cat.numpy(), rc) and np.array_equal(got.reward.numpy(), rrew), t
            pending[0] = (pending[0][0], pending[0][1])
    torch.cuda.synchronize()
    _compare_state(env, ref, 120)
    assert int(env.stats[7].item()) == 0 and int(env.stats[0].item()) == ref.stats[0] > 0


def test_full_size_invariants(D, oracle):
    """BASELINE config 4 slice: 131 072 envs on one GPU.  Size-independent properties + oracle spot checks."""
    B, G, seed = 131072, 4, 7
    perm, lord = D.random_deals(B, seed=1, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, seed=seed, max_actions_per_env=160)
    env.prepare(pd, ld, pool_games=G)
    deck = torch.tensor([4] * 13 + [1, 1], device="cuda")
    sample = np.random.default_rng(0).choice(B, 512, replace=False)
    ref = oracle.RefBatch(len(sample), 2)
    ref.deal(perm.reshape(G, B, 54)[:, sample].reshape(-1, 54), lord.reshape(G, B)[:, sample].reshape(-1), pool_games=G)
    for t in range(130):
        off = env.offsets.to(torch.int64)
        cnt = off[1:] - off[:-1]
        assert (cnt >= 0).all() and int(off[0]) == 0
        assert (cnt[~env.is_done] >= 1).all()
        assert env.num_actions == int(off[B])
        # cards are conserved: hands + everything played == one deck
        total = env.hands().sum(1) + env.taken
        assert (total == deck).all()
        # every listed move fits in the mover's hand
        if t % 20 == 0:
            mv = D.unpack_counts(env.actions_packed)
            owner = torch.repeat_interleave(torch.arange(B, device="cuda"), cnt)
            assert (mv <= env.get_curr_handcards()[owner]).all()
            # spot check against the oracle on the sample
            o_off, o_au, _, o_face = ref.observe(want_f32=False)
            lists = env.actions_packed.cpu().numpy().view(np.uint64)
            offs = off.cpu().numpy()
            got = np.concatenate([lists[offs[b]:offs[b + 1]] for b in sample])
            assert np.array_equal(got, o_au)
            assert np.array_equal(env.face[torch.as_tensor(sample).cuda()].cpu().numpy(), o_face)
        else:
            ref.observe(want_f32=False, want_face=False)
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
        # the oracle sample follows the same Philox stream: env ids are the sampled global ids
        ent = np.array([oracle.philox(seed, int(b), t) for b in sample], dtype=np.uint32)
        ref.step(ent.view(np.int32), mode=1)
        ref.deal(perm.reshape(G, B, 54)[:, sample].reshape(-1, 54), lord.reshape(G, B)[:, sample].reshape(-1),
                 only_done=True, pool_games=G)
    assert int(env.stats[7].item()) == 0
    st = env.stats.cpu().numpy()
    assert st[1] + st[2] + st[3] == st[0] and st[0] > B


def test_full_size_final_states_equal_the_oracle(D, oracle):
    """BASELINE config 4's per-GPU slice, ALL 131 072 envs: 120 fused steps from the deal (two to three games per env,
    re-deals from the pool included), then the complete state of every env and the counters against the oracle's rollout of the same envs
    (ddz_ref_rollout_export, all host threads).  One wrong legal list, index or transition anywhere changes a state."""
    import os
    B, G, seed, K = 131072, 4, 77, 120
    perm, lord = D.random_deals(B, seed=8, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    n, ostats, f, meta = oracle.rollout_export(B, K, 2, seed, perm, lord, G, os.cpu_count() or 1)
    assert n == B * K
    # one chain of launches over all envs
    env = D.BatchedEnvCooperation(B, seed=seed, max_actions_per_env=160)
    env.prepare(pd, ld, pool_games=G)
    for _ in range(K):
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
    ef, emeta = env._fields()
    assert np.array_equal(ef.cpu().numpy().view(np.uint64), f)
    assert np.array_equal(emeta.cpu().numpy().view(np.uint32), meta)
    st = env.stats.cpu().numpy()
    assert np.array_equal(st[[0, 1, 2, 3, 4, 5, 6, 9]], ostats[[0, 1, 2, 3, 4, 5, 6, 9]]) and st[7] == 0
    assert st[8] - env.num_actions == ostats[8]                    # every list the steps consumed, move for move in length
    assert np.median(meta >> 8) >= 2 and (meta >> 8).max() >= 3   # deals consumed: most envs are past their first game
    # the shipped launch shape: four stream-parallel env groups replayed from CUDA graphs
    ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=4, seed=seed, max_actions_per_env=160)
    ge.prepare(pd, ld, pool_games=G)
    ge.capture(steps_per_graph=2)
    for _ in range(K // 2):
        ge.replay()
    ge.join(); torch.cuda.synchronize()
    gf = torch.cat([e._fields()[0] for e in ge.envs], dim=1).cpu().numpy().view(np.uint64)
    gm = torch.cat([e._fields()[1] for e in ge.envs]).cpu().numpy().view(np.uint32)
    assert np.array_equal(gf, f) and np.array_equal(gm, meta)
    assert np.array_equal(ge.stats.cpu().numpy()[[0, 1, 2, 3, 4, 5, 6, 9]], ostats[[0, 1, 2, 3, 4, 5, 6, 9]])


def test_config5_full_size_lists_equal_the_oracle(D, oracle):
    """BASELINE config 5 at the bench's size: the lists of all 131 072 adversarial pairs (18 M moves), list lengths and
    an order-sensitive digest of every move against the oracle's generator -- content AND canonical order, not a sample."""
    n = 131072
    h, l = D.adversarial_pairs(n, seed=12345)
    gen = D.MoveGenerator(n)
    hd = torch.as_tensor(h.view(np.int64)).cuda()
    ld = torch.as_tensor(l.view(np.int64)).cuda()
    acts, offs = gen.generate(hd, ld)
    torch.cuda.synchronize()
    offs = offs.cpu().numpy()
    moves, counts, un, od = oracle.get_moves_digest(h, l)
    assert moves == offs[-1] and moves > 15_000_000
    assert np.array_equal(np.diff(offs), counts)
    gun, god = oracle.lists_digest(acts[:moves].cpu().numpy(), offs)
    assert gun == un and god == od
    assert int(gen.stats[7].item()) == 0


def test_state_prob_getters(D, oracle):
    """get_state_prob (envi.py:94) and get_state_prob_manual (server/core.py:26-33) against the oracle."""
    B = 200
    perm, lord = D.random_deals(B, seed=41)
    env = D.BatchedEnvComplicated(B)
    env.prepare(perm, lord)
    ref = oracle.RefBatch(B, 1)
    ref.deal(perm, lord)
    for t in range(25):
        env.rollout_step()
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=0, env0=0, step=t)
    _, _, _, face = ref.observe(want_f32=False)
    prob = env.get_state_prob().cpu().numpy()
    assert np.array_equal(prob, face[:, 5:].reshape(B, 120))
    # manual form: known = played + own hand, sizes of the two other players (server/core.py:26-33)
    hands = env.hands().cpu().numpy()
    role = (env.get_role_ID() - 1).cpu().numpy()
    taken = env.taken.cpu().numpy()
    for b in range(0, B, 7):
        known = hands[b, role[b]] + taken[b]
        known60 = (np.arange(4)[None, :] < known[:, None]).astype(np.int32).reshape(60)
        s1, s2 = hands[b, (role[b] + 1) % 3].sum(), hands[b, (role[b] + 2) % 3].sum()
        got = D.Env.get_state_prob_manual(known60, s1, s2, device="cuda").cpu().numpy()
        assert np.array_equal(got, oracle.state_prob_manual(known60, s1, s2))
        assert np.array_equal(got, prob[b])


# ------------------------------------------------------------------ batched Q-scoring shim (SURVEY 8f rank 1)
def test_select_actions_kernel(D, oracle):
    rng = np.random.default_rng(2)
    B = 5000
    cnt = rng.integers(0, 40, B)
    cnt[rng.random(B) < 0.1] = 0
    off = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
    q = rng.standard_normal(off[-1]).astype(np.float32)
    q[rng.integers(0, len(q), 2000)] = 0.5          # ties: the FIRST maximum must win, like torch.argmax
    q[rng.integers(0, len(q), 2000)] = 3.0

    class FakeEnv:
        pass
    env = FakeEnv()
    env.B, env.env0, env._stepno = B, 77, 5
    env.offsets = torch.as_tensor(off).cuda()
    pol = D.BatchedGreedyPolicy(None, epsilon=0.0, seed=9)
    got = pol.select(env, torch.as_tensor(q).cuda()).cpu().numpy()
    want = np.array([np.argmax(q[off[b]:off[b + 1]]) if cnt[b] else -1 for b in range(B)])
    assert np.array_equal(got, want)
    pol = D.BatchedGreedyPolicy(None, epsilon=1.0, seed=9)
    got = pol.select(env, torch.as_tensor(q).cuda()).cpu().numpy()
    want = np.array([oracle.philox(9 ^ 0xD1B54A32D192ED03, 77 + b, 5) % cnt[b] if cnt[b] else -1 for b in range(B)])
    assert np.array_equal(got, want)
    pol = D.BatchedGreedyPolicy(None, epsilon=0.3, seed=9)
    got = pol.select(env, torch.as_tensor(q).cuda()).cpu().numpy()
    greedy = np.array([np.argmax(q[off[b]:off[b + 1]]) if cnt[b] else -1 for b in range(B)])
    frac = np.mean((got != greedy)[cnt > 1])
    assert 0.15 < frac < 0.35                        # explores about 30 % of the time (minus lucky draws)


def test_dqn_lord_vs_random_matches_oracle_env(D, oracle):
    """BASELINE config 3 in small: the lord picks argmax_a Q(face, a) with a (random-init) network of the reference's
    contract, the farmers play random legal moves.  The GPU env and the oracle env, driven by the same network, must
    make the same decisions and end with the same win counts (the +-1 pp win-rate criterion, met exactly)."""
    from qnet_like import QNetLike
    torch.manual_seed(0)
    B, G, steps = 1024, 4, 150
    net = QNetLike(9).cuda().eval()
    policy = D.BatchedGreedyPolicy(net)
    perm, lord = D.random_deals(B, seed=23, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, debug=True)
    env.prepare(pd, ld, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    rng = np.random.default_rng(1)
    mism = 0
    for t in range(steps):
        # --- decisions from the GPU env
        is_lord = env.get_role_ID() == 2
        q = policy.q_values(env, is_lord if t % 2 else None)      # masked and unmasked scoring agree on the lord's envs
        greedy = policy.select(env, q)
        off = env.offsets
        cnt = (off[1:] - off[:-1])
        ent = torch.as_tensor(rng.integers(0, 1 << 30, B).astype(np.int32)).cuda()
        choice = torch.where(is_lord, greedy, torch.where(cnt > 0, ent % cnt.clamp(min=1), torch.zeros_like(ent))).to(torch.int32)
        # --- the same decisions recomputed from the ORACLE's features through the same network and the same call pattern
        o_off, o_au, o_af, o_face = ref.observe()
        assert np.array_equal(o_off, off.cpu().numpy())

        class OracleView:                     # quacks like the env for BatchedGreedyPolicy.q_values
            B = env.B
            face = torch.as_tensor(o_face).cuda()
            def valid_actions(self):
                return torch.as_tensor(o_af).cuda(), torch.as_tensor(o_off).cuda()
        q_ref = policy.q_values(OracleView(), is_lord if t % 2 else None)
        qg, qr = q.cpu().numpy(), q_ref.cpu().numpy()
        lord_rows = np.repeat(is_lord.cpu().numpy(), np.diff(o_off))
        assert np.array_equal(qg[lord_rows], qr[lord_rows])       # bit-identical features, same batches -> same Q
        lord_np = is_lord.cpu().numpy()
        greedy_ref = np.array([np.argmax(qr[o_off[b]:o_off[b + 1]]) if o_off[b + 1] > o_off[b] else -1 for b in range(B)])
        mism += int(np.sum((greedy_ref != greedy.cpu().numpy()) & lord_np))
        # --- both envs take the GPU decisions (the action-index stream of the parity contract)
        env.rollout_step(choice, mode=D.native.CHOICE_INDEX, perm=pd, lord_pile=ld, pool_games=G)
        ref.step(choice.cpu().numpy(), mode=0)
        ref.deal(perm, lord, only_done=True, pool_games=G)
    assert mism == 0                                              # identical features -> identical argmax
    _compare_state(env, ref, steps)
    st = env.stats.cpu().numpy()
    assert np.array_equal(st[[0, 1, 2, 3, 4]], ref.stats[[0, 1, 2, 3, 4]]) and st[0] > B
    assert st[7] == 0


def test_grouped_env_trajectories_do_not_depend_on_grouping(D, oracle):
    """GroupedEnv: 2 and 4 stream-parallel groups (eager steps, then CUDA-graph replays) reach exactly the state a
    single batch reaches, because Philox and the deal rows are keyed by the global env id."""
    B, P, seed = 4096, 4, 5
    perm, lord = D.random_deals(B, seed=3, pool_games=P)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    single = D.BatchedEnvCooperation(B, seed=seed)
    single.prepare(pd, ld, pool_games=P)
    steps = 6 + 3 * 8
    for _ in range(steps):
        single.rollout_step(perm=pd, lord_pile=ld, pool_games=P)
    torch.cuda.synchronize()
    want_f, want_m = single._fields()
    for groups in (2, 4):
        ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=groups, seed=seed)
        ge.prepare(perm, lord, pool_games=P)
        for _ in range(6):
            ge.rollout_step()
        ge.capture(steps_per_graph=8)
        for _ in range(3):
            ge.replay()
        ge.join()
        torch.cuda.synchronize()
        f = torch.cat([e._fields()[0] for e in ge.envs], 1)
        m = torch.cat([e._fields()[1] for e in ge.envs])
        assert torch.equal(f, want_f) and torch.equal(m, want_m), groups
        face = torch.cat([e.face for e in ge.envs])
        assert torch.equal(face, single.face)
        keep = [0, 1, 2, 3, 4, 5, 6, 7, 9]
        assert torch.equal(ge.stats[keep], single.stats[keep]) and int(ge.stats[7]) == 0


# ------------------------------------------------------------------ ragged / tiny / multi-wave batches
@pytest.mark.parametrize("B", [1, 31, 33, 100, 1000])
def test_ragged_batch_sizes(D, oracle, B):
    """B not a multiple of the 32-env warp tile (and smaller than one tile): partial warps, partial CTAs."""
    P = 2
    perm, lord = D.random_deals(B, seed=60 + B, pool_games=P)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvComplicated(B, seed=B)
    env.prepare(pd, ld, pool_games=P)
    ref = oracle.RefBatch(B, 1)
    ref.deal(perm, lord, pool_games=P)
    for t in range(70):
        _compare_observation(env, ref, t)
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=P)
        ref.step(mode=2, seed=B, env0=0, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=P)
    _compare_state(env, ref, 70)
    assert int(env.stats[7].item()) == 0


def test_multi_wave_batch_uses_ticket_tiles(D, oracle):
    """300 000 envs = 2344 CTAs, more than fit on the device at once: tiles come from the atomic ticket (start order)
    instead of the launch position, and the look-back chain spans several waves.  Oracle check on a sample + CSR
    invariants over the whole batch."""
    B, P, seed = 300_000, 2, 8
    perm, lord = D.random_deals(B, seed=2, pool_games=P)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnv(B, seed=seed, max_actions_per_env=128)
    env.prepare(pd, ld, pool_games=P)
    sample = np.sort(np.random.default_rng(1).choice(B, 600, replace=False))
    sample[-1] = B - 1
    sample[0] = 0
    ref = oracle.RefBatch(len(sample), 0)
    sp = perm.reshape(P, B, 54)[:, sample].reshape(-1, 54)
    sl = lord.reshape(P, B)[:, sample].reshape(-1)
    ref.deal(sp, sl, pool_games=P)
    st = torch.as_tensor(sample).cuda()
    for t in range(40):
        o_off, o_au, _, o_face = ref.observe(want_f32=False)
        off = env.offsets.to(torch.int64)
        cnt = off[1:] - off[:-1]
        assert int(off[0]) == 0 and (cnt >= 0).all() and env.num_actions == int(off[B])
        assert np.array_equal(cnt[st].cpu().numpy(), np.diff(o_off))
        lists = env.actions_packed
        idx = torch.cat([torch.arange(int(off[b]), int(off[b + 1]), device="cuda") for b in sample[:50]])
        want = np.concatenate([o_au[o_off[i]:o_off[i + 1]] for i in range(50)])
        assert np.array_equal(lists[idx].cpu().numpy().view(np.uint64), want)
        assert np.array_equal(env.face[st].cpu().numpy(), o_face)
        if t % 10 == 0:                                    # every one-hot row is the thermometer of its packed move
            rows = env.valid_actions()[0]
            pick = torch.randint(0, rows.shape[0], (20000,), device="cuda")
            mv = D.unpack_counts(lists[pick])
            thermo = (torch.arange(4, device="cuda")[None, None, :] < mv[:, :, None]).to(torch.float32)
            assert torch.equal(rows[pick], thermo)
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=P)
        ent = np.array([oracle.philox(seed, int(b), t) for b in sample], dtype=np.uint32)
        ref.step(ent.view(np.int32), mode=1)
        ref.deal(sp, sl, only_done=True, pool_games=P)
    assert int(env.stats[7].item()) == 0
    assert int(env.stats[4].item()) == 40 * B


def test_all_envs_finished_and_empty_lists(D):
    """An env that is finished and not re-dealt has no legal move, ignores steps, and still encodes a face."""
    B = 64
    perm, lord = D.random_deals(B, seed=4)
    env = D.BatchedEnvCooperation(B, debug=True)
    env.prepare(perm, lord)
    for _ in range(400):                                   # no re-deal: every game runs to its end and stays there
        env.rollout_step()
    assert env.is_done.all()
    assert env.num_actions == 0 and int(env.offsets[B]) == 0
    before = env._state.clone()
    r, done, cat = env.rollout_step()
    assert torch.equal(env._state, before) and (cat == -1).all() and (r == 0).all() and done.all()
    assert torch.isfinite(env.face).all() and env.face.shape == (B, 9, 15, 4)
    st = env.stats.cpu().numpy()
    assert st[0] == B and st[1] + st[2] + st[3] == B and st[7] == 0


def test_payload_ingest_matches_reference_predictor(D, golden):
    """SURVEY 8f rank 3: payloads in the wire format of server/client.py -> device state -> face / valid_actions equal to
    what the reference's own Predictor.face / Predictor.valid_actions (server/core.py:26-67) computed for them."""
    g = golden.core_payloads
    env = D.env_from_arrays(g["role"], g["hand"], g["history"], g["last_taken"], g["left"], debug=True)
    assert np.array_equal(env.face.cpu().numpy(), g["face"])
    acts, offs = env.valid_actions()
    assert np.array_equal(offs.cpu().numpy().astype(np.int64), g["actions_off"])
    assert np.array_equal(acts.cpu().numpy(), g["actions"])
    # and through the dict form of the wire format
    def cards(c):
        return [r + 3 for r in range(15) for _ in range(int(c[r]))]
    payloads = [{"role_id": int(g["role"][b]), "cur_cards": cards(g["hand"][b]),
                 "history": {q: cards(g["history"][b, q]) for q in range(3)},
                 "last_taken": {str(q): cards(g["last_taken"][b, q]) for q in range(3)},
                 "left": {q: int(g["left"][b, q]) for q in range(3)}} for b in range(40)]
    env2 = D.env_from_payloads(payloads)
    assert np.array_equal(env2.face.cpu().numpy(), g["face"][:40])
    with pytest.raises(ValueError):
        D.env_from_arrays([3], g["hand"][:1], g["history"][:1], g["last_taken"][:1], g["left"][:1])


def test_config1_thousand_seeded_games_same_winners_as_oracle(D, oracle):
    """BASELINE config 1/2 cross-check: the 1000 games of the documented default deal stream, random play from the Philox
    stream, run to the end on the GPU env and on the oracle: same winner in every game, same number of decisions."""
    n = 1000
    env = D.BatchedEnv(n, seed=20260101)
    env.prepare()                                   # no arguments: default_deals(0, n)
    perm, lord = D.default_deals(0, n)
    ref = oracle.RefBatch(n, 0)
    ref.deal(perm, lord)
    for t in range(200):
        env.rollout_step()
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=20260101, env0=0, step=t)
    assert env.is_done.all() and ref.envs["done"].all()
    assert np.array_equal(env.winner.cpu().numpy(), ref.envs["winner"])
    st = env.stats.cpu().numpy()
    assert np.array_equal(st[[0, 1, 2, 3, 4, 9]], ref.stats[[0, 1, 2, 3, 4, 9]]) and st[0] == n


# ------------------------------------------------------------------ trainer driver pieces (SURVEY 8f rank 2)
def test_transition_assembly_matches_reference_game_loop(D, oracle, golden):
    """TransitionCollector vs the perceive() calls the UNMODIFIED game.py (Game.play, lord in training, all seats driven by
    a recorded index stream) made on the same 40 deals: same (s0, a0, r, s1, a1, done), game by game, in order."""
    g = golden.game_transitions
    seed, perms = int(g["seed"]), g["perms"]
    B = len(perms)
    env = D.BatchedEnvCooperation(B, debug=True)
    env.prepare(perms, np.zeros(B, np.int8))
    col = D.TransitionCollector(env, role=1, reward=100.0)
    got = [[] for _ in range(B)]

    def take(out):
        s0, a0, r, s1, a1, done, idx = (x.cpu().numpy() for x in out)
        for i, b in enumerate(idx):
            got[b].append((s0[i], a0[i], float(r[i]), s1[i], a1[i], bool(done[i])))

    for t in range(200):
        acts, offs = env.valid_actions()
        off = offs.cpu().numpy().astype(np.int64)
        cnt = np.diff(off)
        k0 = np.array([oracle.philox(seed, b, 2 * t) % cnt[b] if cnt[b] else 0 for b in range(B)])
        k1 = np.array([oracle.philox(seed, b, 2 * t + 1) % cnt[b] if cnt[b] else 0 for b in range(B)])
        live = torch.as_tensor(cnt > 0).cuda()[:, None, None]
        rows0 = acts[torch.as_tensor(np.minimum(off[:-1] + k0, max(off[-1] - 1, 0))).cuda()] * live
        rows1 = acts[torch.as_tensor(np.minimum(off[:-1] + k1, max(off[-1] - 1, 0))).cuda()] * live
        take(col.on_turn(rows0, rows1))
        was_done = env.is_done.clone()
        env.step(k0.astype(np.int32))
        env.observe()
        take(col.on_step_done(env.is_done & ~was_done))
        if bool(env.is_done.all()):
            break
    assert bool(env.is_done.all())
    n = 0
    for b in range(B):
        rows = np.flatnonzero(g["game"] == b)
        assert len(got[b]) == len(rows), (b, len(got[b]), len(rows))
        for j, row in enumerate(rows):
            s0, a0, r, s1, a1, done = got[b][j]
            assert np.array_equal(s0, g["s0"][row]) and np.array_equal(a0, g["a0"][row]), (b, j)
            assert r == g["r"][row] and done == bool(g["done"][row]), (b, j)
            assert np.array_equal(s1, g["s1"][row]) and np.array_equal(a1, g["a1"][row]), (b, j)
            n += 1
    assert n == len(g["game"]) > 300
    st = env.stats.cpu().numpy()
    assert st[1] == int(g["lord_wins"]) and st[2] + st[3] == int(g["farmer_wins"])


def test_replay_buffer_and_td_step(D):
    from qnet_like import QNetLike
    torch.manual_seed(0)
    dev = torch.device("cuda")
    rb = D.ReplayBuffer(100, 9, dev)
    mk = lambda n, base: (torch.full((n, 9, 15, 4), base, device=dev), torch.full((n, 15, 4), base, device=dev),
                          torch.full((n,), base, device=dev), torch.full((n, 9, 15, 4), base + 0.5, device=dev),
                          torch.zeros((n, 15, 4), device=dev), torch.zeros(n, device=dev))
    rb.append(*mk(60, 1.0))
    assert len(rb) == 60
    rb.append(*mk(70, 2.0))                          # wraps: the 30 oldest entries are overwritten, like deque(maxlen)
    assert len(rb) == 100
    assert int((rb.r == 1.0).sum()) == 30 and int((rb.r == 2.0).sum()) == 70
    batch = rb.sample(32)
    assert batch[0].shape == (32, 9, 15, 4) and batch[2].shape == (32, 1)
    # td_step == the reference's arithmetic (dqn.py:39-47)
    policy, target = QNetLike(9).to(dev), QNetLike(9).to(dev)
    target.load_state_dict(policy.state_dict())
    opt = torch.optim.Adam(policy.parameters(), 1e-3)
    s0, a0, r, s1, a1, done = (torch.rand(64, 9, 15, 4, device=dev), torch.rand(64, 15, 4, device=dev).round(),
                               torch.randn(64, 1, device=dev), torch.rand(64, 9, 15, 4, device=dev),
                               torch.rand(64, 15, 4, device=dev).round(), (torch.rand(64, 1, device=dev) < 0.3).float())
    with torch.no_grad():
        want = torch.nn.MSELoss()(r + (1 - done) * 0.95 * target(s1, a1), policy(s0, a0))
    first = D.td_step(policy, target, opt, (s0, a0, r, s1, a1, done), 0.95)
    assert torch.allclose(first, want, rtol=1e-5)
    for _ in range(30):
        last = D.td_step(policy, target, opt, (s0, a0, r, s1, a1, done), 0.95)
    assert last < first


# ------------------------------------------------------------------ k-th move in closed form + random playouts (8f rank 4)
def test_kth_moves_equal_the_enumerated_lists(D, oracle, golden):
    """select_legal: the idx-th move computed from counts + unranking == the idx-th entry of the enumerated list, for
    every index of every golden / adversarial / random (hand, last) pair."""
    g = golden.legal_sets
    rng = np.random.default_rng(17)
    hands = np.concatenate([g["hands"], _rand_hands(rng, 1500)])
    z = np.zeros(15, np.int8)
    lasts = [l for l in g["lasts"]]
    for i in range(1500):
        if i % 2:
            om = oracle.get_moves(_rand_hands(rng, 1, 2, 21)[0], z, fast=True)
            lasts.append(om[rng.integers(len(om))])
        else:
            lasts.append(z)
    lasts = np.array(lasts, np.int8)
    packed, offsets = D.get_moves(hands, lasts)
    packed, off = packed.cpu().numpy(), offsets.cpu().numpy().astype(np.int64)
    owner = np.repeat(np.arange(len(hands)), np.diff(off))
    idx = np.arange(len(packed)) - off[owner]
    got, cnt = D.kth_moves(hands[owner], lasts[owner], idx)
    assert np.array_equal(got.cpu().numpy(), packed)
    assert np.array_equal(cnt.cpu().numpy(), np.diff(off)[owner])
    bad, _ = D.kth_moves(hands[:100], lasts[:100], np.diff(off)[:100])          # one past the end
    assert (bad.cpu().numpy() == -1).all()


def test_playout_equals_step_by_step_rollout(D, oracle):
    """ddz_playout (one launch, no lists) == stepping the same envs move by move with the same Philox stream: the MCTS
    default policy (server/mcts/default_policy.py:4-10) as a primitive."""
    B, seed = 3000, 31337
    perm, lord = D.random_deals(B, seed=15)
    env = D.BatchedEnv(B, seed=seed, env0=500)
    env.prepare(perm, lord)
    for _ in range(7):                                   # start from mid-game positions, step counter at 7
        env.rollout_step()
    ref = oracle.RefBatch(B, 0)
    ref.deal(perm, lord)
    for t in range(7):
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=seed, env0=500, step=t)
    _compare_state(env, ref, 7)
    steps = env.playout(max_steps=20)                    # a bounded playout first ...
    taken = np.zeros(B, np.int64)
    for t in range(7, 27):
        ref.observe(want_f32=False, want_face=False)
        before = ref.envs["done"].copy()
        ref.step(mode=2, seed=seed, env0=500, step=t)
        taken += (before == 0)
    _compare_state(env, ref, 27)
    assert np.array_equal(steps.cpu().numpy(), taken)
    env.playout(max_steps=300)                           # ... then to the end of every game
    for t in range(27, 327):
        ref.observe(want_f32=False, want_face=False)
        ref.step(mode=2, seed=seed, env0=500, step=t)
        if ref.envs["done"].all():
            break
    assert env.is_done.all()
    assert np.array_equal(env.winner.cpu().numpy(), ref.envs["winner"])
    _f, _m = ref.export()
    assert np.array_equal(env._fields()[0].cpu().numpy().view(np.uint64), _f)
    st = env.stats.cpu().numpy()
    assert np.array_equal(st[[0, 1, 2, 3, 4, 5, 6, 9]], ref.stats[[0, 1, 2, 3, 4, 5, 6, 9]]) and st[7] == 0


def test_mcts_moves_match_get_moves_py(D, oracle, golden):
    """ddz_mcts_moves == the unmodified server/mcts/get_moves.py on the golden positions (filter, value, stable sort,
    lowest/highest interleave), and == the oracle's restatement on random and adversarial pairs."""
    g = golden.mcts_moves
    offs = g["offsets"]
    lists, counts = D.mcts_moves(g["hands"], g["lasts"])
    lists, counts = lists.cpu().numpy().view(np.uint64), counts.cpu().numpy()
    assert np.array_equal(counts, np.diff(offs))
    for i in range(len(counts)):
        assert np.array_equal(oracle.unpack(lists[i, :counts[i]]), g["moves"][offs[i]:offs[i + 1]]), i
    rng = np.random.default_rng(23)
    hands = _rand_hands(rng, 600, 1, 21)
    z = np.zeros(15, np.int8)
    lasts = []
    for i in range(600):
        om = oracle.get_moves(_rand_hands(rng, 1, 2, 21)[0], z, fast=True)
        lasts.append(om[rng.integers(len(om))] if i % 2 else z)
    ah, al = D.adversarial_pairs(256, seed=9)
    hands = np.concatenate([hands, oracle.unpack(ah)])
    lasts = np.concatenate([np.array(lasts, np.int8), oracle.unpack(al)])
    lists, counts = D.mcts_moves(hands, lasts)
    lists, counts = lists.cpu().numpy().view(np.uint64), counts.cpu().numpy()
    pruned = 0
    for i in range(len(hands)):
        want = oracle.mcts_moves(hands[i], lasts[i])
        assert counts[i] == len(want) and np.array_equal(oracle.unpack(lists[i, :counts[i]]), want), i
        pruned += len(want) > 10
    assert pruned > 200


def test_search_policy_playout_equals_oracle(D, oracle):
    """ddz_playout_pruned: every decision is entry  philox % len  of the bot's pruned move list (tree.py:83-91 over
    get_moves.py:36-69) -- the same games, move for move, as the oracle driven with that policy."""
    from uct_reference_algorithm import pruned_playout_step
    B, seed = 384, 99
    perm, lord = D.random_deals(B, seed=21)
    env = D.BatchedEnv(B, seed=seed, env0=40)
    env.prepare(perm, lord)
    ref = oracle.RefBatch(B, 0)
    ref.deal(perm, lord)
    steps = env.playout(max_steps=9, policy="search")    # from the deal: the long lists, all pruned
    for t in range(9):
        pruned_playout_step(oracle, ref, seed, 40, t)
    _compare_state(env, ref, 9)
    assert (steps.cpu().numpy() == 9).all()
    uni = D.BatchedEnv(B, seed=seed, env0=40)
    uni.prepare(perm, lord)
    uni.playout(max_steps=9)                             # the uniform policy plays different games
    assert not torch.equal(uni._fields()[0], env._fields()[0])
    env.playout(max_steps=300, policy="search")
    for t in range(9, 309):
        pruned_playout_step(oracle, ref, seed, 40, t)
        if ref.envs["done"].all():
            break
    assert env.is_done.all()
    assert np.array_equal(env.winner.cpu().numpy(), ref.envs["winner"])
    _f, _m = ref.export()
    assert np.array_equal(env._fields()[0].cpu().numpy().view(np.uint64), _f)
    st = env.stats.cpu().numpy()
    assert np.array_equal(st[[0, 1, 2, 3, 4, 9]], ref.stats[[0, 1, 2, 3, 4, 9]]) and st[7] == 0


def test_flat_monte_carlo_move_evaluation(D, oracle):
    """evaluate_moves (the MCTS bot's job with playouts instead of a tree): a move that empties the hand wins every
    playout; win rates agree with playouts stepped on the oracle within sampling noise."""
    z = np.zeros(15, np.int64)
    hands = np.zeros((3, 15), np.int64)
    hands[1, [0, 1, 2, 3, 4]] = 1          # lord: 3 4 5 6 7  -> the straight ends the game at once
    hands[2, [5, 5 + 1]] = 2               # down: 88 99
    hands[0, [10, 11, 12]] = [1, 2, 1]     # up:   K AA 2
    hist = np.zeros((3, 15), np.int64)
    moves, win = D.evaluate_moves(1, hands, hist, np.zeros((3, 15), np.int64), sims=512, seed=5)
    straight = np.array([1] * 5 + [0] * 10)
    i = int(np.flatnonzero((moves == straight).all(1))[0])
    assert win[i] == 1.0 and len(moves) == 6                 # five singles + the straight
    assert (win[np.arange(len(moves)) != i] < 1.0).all()
    # cross-check one move's win rate against the oracle driven with its own random stream
    j = 0
    rng = np.random.default_rng(0)
    wins, n = 0, 400
    for _ in range(n):
        rb = oracle.RefBatch(1, 0)
        rb.envs["hand"][0] = hands
        rb.envs["cur"] = 1
        first = True
        while not rb.envs["done"][0]:
            off, _, _, _ = rb.observe(want_f32=False, want_face=False)
            k = j if first else int(rng.integers(off[1]))
            first = False
            rb.step(np.array([k], np.int32), mode=0)
        wins += int(rb.envs["winner"][0] == 1)
    assert abs(wins / n - win[j]) < 0.09                     # 3 sigma of two binomial estimates


def test_step_manual_rejects_a_move_that_is_not_legal(D):
    """envi.py:63-70 step_manual with a one-hot that is not among valid_actions(): refused, flagged, state untouched."""
    B = 32
    perm, lord = D.random_deals(B, seed=77)
    env = D.BatchedEnv(B)
    env.prepare(perm, lord)
    before = env._state.clone()
    acts, offs = env.valid_actions()
    bogus = torch.zeros((B, 15, 4), device="cuda")
    bogus[:, 0, :] = 1                                   # four 3s: nobody holds them all in (almost) every deal
    has_bomb3 = env.get_curr_handcards()[:, 0] == 4
    r, done, cat = env.step_manual(bogus)
    torch.cuda.synchronize()
    bad = ~has_bomb3
    assert bad.any()
    assert (cat[bad] == -1).all() and (r[bad] == 0).all()
    f_before = before[: 18 * B].view(torch.int64).view(9, B)
    assert torch.equal(env._fields()[0][:, bad], f_before[:, bad])
    assert (((env._fields()[1] >> 5) & 1).bool() == bad).all()
    assert int(env.stats[7].item()) == int(bad.sum())
    # the B = 1 view: a legal random move from host entropy works as in the reference (envi.py:79-85)
    one = D.Env(debug=True)
    one.reset(); one.prepare()
    n = one.valid_actions().shape[0]
    r1, d1, c1 = one.step_random(12345)
    assert (r1, d1) == (0, False) and 1 <= c1 <= 14 and n > 0 and one.get_role_ID() == 3


def test_legal_move_counts_at_scale(D, oracle):
    """400 000 random (hand, last) pairs through ddz_legal_moves: the list lengths equal the oracle's, the kernel's own
    closed-form-count == enumerated-count self-check never fires, every list is duplicate-free, sorted into the canonical
    category order, and fits in the hand."""
    rng = np.random.default_rng(2024)
    n = 400_000
    deck = np.array([i // 4 for i in range(52)] + [13, 14])
    sizes = rng.integers(1, 21, n)
    order = np.argsort(rng.random((n, 54)), axis=1)                      # a random deal per row
    hands = np.zeros((n, 15), np.int8)
    ranks = deck[order]
    for k in range(20):
        take = sizes > k
        np.add.at(hands, (np.flatnonzero(take), ranks[take, k]), 1)
    # previous moves: legal lead moves of other random hands (computed on the GPU), half of the pairs lead
    other = np.zeros((n, 15), np.int8)
    for k in range(17):
        np.add.at(other, (np.arange(n), ranks[:, 30 + k]), 1)
    lead_lists, lead_off = D.get_moves(other, np.zeros_like(other))
    lo = lead_off.cpu().numpy().astype(np.int64)
    pick = lo[:-1] + (rng.integers(0, 1 << 30, n) % np.diff(lo))
    lasts_packed = lead_lists[torch.as_tensor(pick).cuda()].clone()
    lasts_packed[torch.as_tensor(rng.random(n) < 0.5).cuda()] = 0
    gen = D.MoveGenerator(n)
    hp = D.pack_counts(torch.as_tensor(hands).cuda()).contiguous()
    acts, offs = gen.generate(hp, lasts_packed)
    torch.cuda.synchronize()
    assert int(gen.stats[7].item()) == 0                                  # count_legal == what the walks emitted
    off = offs.to(torch.int64)
    cnt = (off[1:] - off[:-1]).cpu().numpy()
    lasts = D.unpack_counts(lasts_packed).cpu().numpy().astype(np.int8)
    sample = rng.choice(n, 60_000, replace=False)
    assert np.array_equal(cnt[sample], oracle.count_moves_batch(hands[sample], lasts[sample]))
    total = int(off[n])
    mv = acts[:total]
    owner = torch.repeat_interleave(torch.arange(n, device="cuda"), off[1:] - off[:-1])
    counts = D.unpack_counts(mv)
    assert (counts <= torch.as_tensor(hands).cuda().to(torch.int64)[owner]).all()                 # containment
    same_owner = owner[1:] == owner[:-1]
    assert (mv[1:][same_owner] != mv[:-1][same_owner]).all()                                     # no immediate repeats
    key = owner * (1 << 20) + torch.arange(total, device="cuda")                                 # (sanity of CSR order)
    assert (key[1:] > key[:-1]).all()
    uniq = torch.unique(torch.stack([owner, mv], 1), dim=0).shape[0]
    assert uniq == total                                                                         # duplicate-free lists


@pytest.mark.parametrize("cls,variant,use_entropy", [("BatchedEnvCooperation", 2, False), ("BatchedEnv", 0, True),
                                                     ("BatchedEnvComplicated", 1, False),
                                                     ("BatchedEnvCooperationSimplify", 3, True)])
def test_multi_step_launch_bit_exact(D, oracle, cls, variant, use_entropy):
    """ddz_rollout_steps: K env-steps per native call == K single steps of the oracle, every slice of the trajectory
    (lists, one-hots, face, results) and the final state, over several calls with re-deals."""
    B, G, K, seed, launches = 2048 + 37, 4, 12, 77, 9
    rng = np.random.default_rng(5)
    perm, lord = D.random_deals(B, seed=15, pool_games=G)
    perm_d, lord_d = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = getattr(D, cls)(B, seed=seed, env0=300, max_actions_per_env=128)
    env.prepare(perm_d, lord_d, pool_games=G)
    ref = oracle.RefBatch(B, variant)
    ref.deal(perm, lord, pool_games=G)
    traj = D.Trajectory(env, K)
    t = 0
    for it in range(launches):
        ent = rng.integers(0, 1 << 31, (K, B)).astype(np.int32) if use_entropy else None
        env.rollout_steps(traj, entropy=ent, perm=perm_d, lord_pile=lord_d, pool_games=G)
        torch.cuda.synchronize()
        offs = traj.offsets.cpu().numpy()
        for s in range(K):
            ref.observe(want_f32=False)                     # the oracle steps from its current lists
            if use_entropy:
                rr, rd, rc, rrew = ref.step(mode=1, choice=ent[s])
            else:
                rr, rd, rc, rrew = ref.step(mode=2, seed=seed, env0=300, step=t)
            ref.deal(perm, lord, only_done=True, pool_games=G)
            t += 1
            off, au, af, face = ref.observe(want_f32=(s % 5 == 0))
            n = int(off[B])
            assert np.array_equal(offs[s], off), (it, s)
            assert np.array_equal(traj.actions_u64[s, :n].cpu().numpy().view(np.uint64), au), (it, s)
            assert np.array_equal(traj.face[s].cpu().numpy(), face), (it, s)
            if s % 5 == 0:
                assert np.array_equal(traj.actions_f32[s, :n].cpu().numpy(), af), (it, s)
            assert np.array_equal(traj.r[s].cpu().numpy(), rr) and np.array_equal(traj.done[s].cpu().numpy(), rd), (it, s)
            assert np.array_equal(traj.cat[s].cpu().numpy(), rc) and np.array_equal(traj.reward[s].cpu().numpy(), rrew), (it, s)
        _compare_state(env, ref, t)
    stats = env.stats.cpu().numpy()
    assert stats[7] == 0 and np.array_equal(stats[[0, 1, 2, 3, 4, 5, 6, 9]], ref.stats[[0, 1, 2, 3, 4, 5, 6, 9]])
    # the env carries on with the single-step API from where the launch left it
    n = _compare_observation(env, ref, t)
    assert n > 0
    env.rollout_step(mode=D.native.CHOICE_PHILOX, perm=perm_d, lord_pile=lord_d, pool_games=G)
    ref.step(mode=2, seed=seed, env0=300, step=t)
    ref.deal(perm, lord, only_done=True, pool_games=G)
    _compare_observation(env, ref, t + 1)


def test_multi_step_launch_equals_playout(D, oracle):
    """40 steps per call without re-deal (finished envs stay finished): final state + counters equal a playout of the
    same Philox stream."""
    B, K = 4800, 40
    perm, lord = D.random_deals(B, seed=3)
    a = D.BatchedEnv(B, seed=9, max_actions_per_env=128)
    b = D.BatchedEnv(B, seed=9)
    for e in (a, b):
        e.prepare(perm, lord)
    traj = D.Trajectory(a, K)
    a.rollout_steps(traj)
    b.playout(K)
    torch.cuda.synchronize()
    fa, ma = a._fields(); fb, mb = b._fields()
    assert torch.equal(fa, fb) and torch.equal(ma, mb)
    sa, sb = a.stats.cpu().numpy(), b.stats.cpu().numpy()
    assert sa[7] == 0 and np.array_equal(sa[[0, 1, 2, 3, 4, 5, 6, 9]], sb[[0, 1, 2, 3, 4, 5, 6, 9]])
    # the last slice is the observation of the final state
    a.observe()
    assert torch.equal(traj.offsets[K - 1], a.offsets)
    n = int(a.offsets[B].item())
    assert torch.equal(traj.actions_u64[K - 1, :n], a.actions_packed) and torch.equal(traj.face[K - 1], a.face)


def test_overflowing_lists_are_safe(D, oracle):
    """cap smaller than the total: the tail of the lists is dropped and stats[7] says so -- never an out-of-bounds access --
    and no env is lost: cut lists are played from their visible part, envs whose list was dropped sit the step out WITHOUT a
    sticky error and move again once their list fits; asking for the lists grows the buffers and observes again."""
    B, G = 8192, 2
    perm, lord = D.random_deals(B, seed=21, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, seed=2, max_actions_per_env=8)        # 20-card leads have far more than 8 moves
    env.prepare(pd, ld, pool_games=G)
    env.observe()
    torch.cuda.synchronize()
    assert int(env.stats[7].item()) >= 1 and int(env.offsets[B].item()) > env.cap
    deck = np.array([4] * 13 + [1, 1])
    waited = 0
    for t in range(300):
        before = int(env.stats[4].item())
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
        waited += B - (int(env.stats[4].item()) - before)
    torch.cuda.synchronize()
    f, meta = env._fields()
    meta = meta.cpu().numpy().view(np.uint32)
    assert ((meta >> 5) & 1).sum() == 0                                     # nobody was stopped for good
    assert waited > 0                                                       # some envs did sit steps out ...
    assert (meta >> 8).min() >= 2                                           # ... but every env finished games and was re-dealt
    cards = D.unpack_counts(f[0:6].t().contiguous()).sum(1).cpu().numpy()   # hands + everything played = one deck, always
    assert (cards == deck).all()
    fresh = D.BatchedEnvCooperation(B, seed=2, max_actions_per_env=8)
    fresh.prepare(pd, ld, pool_games=G)
    ref0 = oracle.RefBatch(B, 2)
    ref0.deal(perm, lord, pool_games=G)
    n = _compare_observation(fresh, ref0, 0)                                # grows the buffers, re-observes: complete lists
    assert fresh.cap >= n > 8 * B


def test_ticket_tiles_with_a_concurrent_kernel(D, oracle):
    """Other kernels share the GPU with the env launches (BASELINE config 3: the Q-network): with ddz_set_tile_order(ticket)
    nothing depends on the env grid being co-resident.  A matmul loop runs on another stream while two env groups step;
    results equal the oracle's and no look-back ever times out (stats[7] == 0).  The default order is checked the same way."""
    B, P = 32768, 2
    perm, lord = D.random_deals(B, seed=9, pool_games=P)
    pr = perm.reshape(P, B, 54)[:, :2048].reshape(-1, 54); lr = lord.reshape(P, B)[:, :2048].reshape(-1)
    for mode in ("ticket", "auto"):
        prev = D.native.set_tile_order(mode)
        try:
            ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=2, seed=6, max_actions_per_env=160)
            ge.prepare(perm, lord, pool_games=P)
            ref = oracle.RefBatch(2048, 2)                                 # the oracle follows the first 2048 envs
            ref.deal(pr, lr, pool_games=P)
            side = torch.cuda.Stream()
            a = torch.randn(4096, 4096, device="cuda")
            for t in range(30):
                with torch.cuda.stream(side):
                    for _ in range(2):
                        a = (a @ a).clamp_(-1, 1)                           # keeps every SM busy next to the env launches
                ge.rollout_step()
                ref.observe(want_f32=False, want_face=False)
                ref.step(mode=2, seed=6, env0=0, step=t)
                ref.deal(pr, lr, only_done=True, pool_games=P)
            ge.join()
            torch.cuda.synchronize()
            assert int(ge.stats[7].item()) == 0, mode
            f, meta = ref.export()
            ef, em = ge.envs[0]._fields()
            assert np.array_equal(ef[:, :2048].cpu().numpy().view(np.uint64), f), mode
            assert np.array_equal(em[:2048].cpu().numpy().view(np.uint32), meta), mode
        finally:
            D.native.set_tile_order(prev)
    assert D.native.set_tile_order("auto") == "auto"


def test_batched_game_trains_and_competes(D):
    """BatchedGame / BatchedDQN (game.py:10-275, dqn.py:10-80 over a batched env): counters agree with the env's own,
    transitions reach the replay buffer, TD steps run, schedules tick; compete() plays the trained net greedily."""
    from qnet_like import QNetLike
    net = lambda: QNetLike(9, width=16)
    roles = {"lord": net, "down": net, "up": None}
    dqns = {"lord": D.BatchedDQN, "down": D.BatchedDQN, "up": None}
    torch.manual_seed(0)
    game = D.BatchedGame(D.BatchedEnvCooperation, roles, dqns, reward_dict={"lord": 100, "down": 50, "up": 50},
                         train_dict={"lord": True, "down": True, "up": False}, seed=3, num_envs=512)
    hist = game.train(1200, log_every=400)
    st = game.env.stats.cpu().numpy()
    assert game.episodes >= 1200 and game.episodes == st[0] and st[7] == 0
    assert (game.lord_total_wins, game.down_total_wins, game.up_total_wins) == (st[1], st[2], st[3])
    assert len(hist) >= 2 and abs(sum(hist[-1][r]["total_win"] for r in ("up", "lord", "down")) - 1.0) < 1e-9
    for role in ("lord", "down"):
        agent = getattr(game, role)
        assert len(agent.replay_buffer) > agent.batch_size and agent.epsilon < 0.5
        rb = agent.replay_buffer
        n = len(rb)
        term = rb.done[:n, 0] == 1
        assert term.any() and (~term).any()
        want = 100.0 if role == "lord" else 50.0
        assert (rb.r[:n, 0][term].abs() == want).all() and (rb.r[:n, 0][~term] == 0).all()
        assert (rb.a1[:n][term] == 0).all()                                   # game.py:123-124: a1 = zeros at the end
        assert (rb.a0[:n].flatten(1).sum(1) >= 0).all() and rb.s0[:n].isfinite().all()
    assert any(h["lord"]["mean_loss"] > 0 for h in hist)
    wins = D.BatchedGame.compete(D.BatchedEnvCooperation, {"lord": net, "down": None, "up": None},
                                 {"lord": D.BatchedDQN, "down": None, "up": None}, None, total=500, debug=False,
                                 num_envs=256, seed=5, nets={"lord": game.lord.policy_net})
    assert sum(wins.values()) >= 500 and wins["lord"] > 0


def test_single_env_view_bookkeeping(D, capsys):
    """envi.py:27,38-61,159-161: old_cards, cards2str and the debug narration of the B = 1 view."""
    env = D.EnvCooperation(debug=True)
    env.reset()
    env.prepare()
    assert env.cards2str([3, 10, 11, 15, 16, 17]) == ["3", "10", "J", "2", "小", "大"]
    hand = list(env.get_curr_handcards())
    acts = env.valid_actions()
    r, done, cat = env.step_manual(acts[0])
    assert list(env.old_cards[1]) == hand and len(hand) == 20          # the landlord moved first
    played = env.onehot2arr(acts[0])
    assert env.left[1] == 20 - int(np.sum(played))
    out = capsys.readouterr().out
    assert "地主出牌" in out and "分别剩余" in out
    env.step_random()
    assert 2 in env.old_cards and len(env.old_cards[2]) == 17
    env.reset()
    assert env.old_cards == {}


@pytest.mark.parametrize("cls", ["BatchedEnv", "BatchedEnvComplicated", "BatchedEnvCooperation", "BatchedEnvCooperationSimplify"])
def test_state_action_encoder(D, cls):
    """ddz_encode_state_actions == torch.cat((face.repeat per action, action), 1) of net.py:81-90, bit for bit, for all
    moves and for the moves of a subset of envs; the Q-scoring shim gives the same values through either input form."""
    from qnet_like import QNetLike
    B = 3000
    perm, lord = D.random_deals(B, seed=31)
    env = getattr(D, cls)(B, seed=4)
    env.prepare(perm, lord)
    for _ in range(25):
        env.rollout_step()
    face = env.face
    acts, offs = env.valid_actions()
    cnt = (offs[1:] - offs[:-1]).to(torch.int64)
    owner = torch.repeat_interleave(torch.arange(B, device="cuda"), cnt)
    want = torch.cat((face[owner], acts.unsqueeze(1)), dim=1)
    x, rows = env.state_actions()
    assert rows is None and torch.equal(x, want)
    mask = (env.get_role_ID() == 2) | (torch.arange(B, device="cuda") % 7 == 0)
    xs, rows = env.state_actions(mask)
    assert torch.equal(rows, mask[owner].nonzero(as_tuple=True)[0]) and torch.equal(xs, want[rows])
    none = torch.zeros(B, dtype=torch.bool, device="cuda")
    assert env.state_actions(none)[0].shape[0] == 0
    torch.manual_seed(1)
    net = QNetLike(env.C, width=8).cuda().eval()

    class TwoInput(torch.nn.Module):                      # the same network without the concatenated entry point
        def __init__(self, inner):
            super().__init__()
            self.inner = inner

        def forward(self, face, actions):
            return self.inner(face, actions)

    qa = D.BatchedGreedyPolicy(net, chunk_actions=4096).q_values(env, mask)
    qb = D.BatchedGreedyPolicy(TwoInput(net), chunk_actions=4096).q_values(env, mask)
    assert torch.equal(qa, qb)


def test_mcts_entry_point(D):
    """mcts(payload) (server/mcts/interface.py:15-45): the search bot's wire format in, a move as card values out."""
    payload = {"role_id": 1,
               "hand_card": {0: [13, 14, 14, 15], 1: [3, 4, 5, 6, 7], 2: [8, 8, 9, 9]},
               "last_taken": {0: [], 1: [], 2: []}}
    assert D.mcts(payload, computation_budget=600) == [3, 4, 5, 6, 7]       # the straight wins on the spot
    # following a pair of 9s with 10 10 J in hand against opponents that are one move from going out: play the 10s
    payload = {"role_id": "2", "hand_card": {"0": [3], "1": [4], "2": [10, 10, 11]},
               "last_taken": {"0": [], "1": [9, 9], "2": []}}
    payload["role_id"] = 2
    assert D.mcts(payload, computation_budget=2000, seed=3) == [10, 10]


def test_deferred_pool_refill(D):
    """HostRollout.refill uploads in the background; the slot is replaced (whole, between two steps) by the first step
    that finds the upload complete, or at once by flush()."""
    B, G = 4096, 4
    perm, lord = D.random_deals(B, seed=1, pool_games=G)
    env = D.BatchedEnvCooperation(B, seed=3)
    env.prepare(perm, lord, pool_games=G)
    host = D.HostRollout(env, perm, lord, G)
    ent = torch.as_tensor(np.random.default_rng(0).integers(0, 1 << 31, B).astype(np.int32)).pin_memory()
    p2, l2 = D.random_deals(B, seed=77)
    p2t, l2t = torch.as_tensor(p2).pin_memory(), torch.as_tensor(l2).pin_memory()
    old = host.perm_d[2].clone()
    host.refill(2, p2t, l2t)
    for _ in range(200):                                  # the upload (220 KB) lands within a few steps
        res = host.step(ent)
        slot = host.perm_d[2].cpu()
        assert torch.equal(slot, old.cpu()) or torch.equal(slot, p2t)      # never a mixture
        if torch.equal(slot, p2t):
            break
    D.HostRollout.wait(res)
    torch.cuda.synchronize()
    assert torch.equal(host.perm_d[2].cpu(), p2t) and torch.equal(host.lord_d[2].cpu(), l2t)
    p3, l3 = D.random_deals(B, seed=78)
    p3t, l3t = torch.as_tensor(p3).pin_memory(), torch.as_tensor(l3).pin_memory()
    host.refill(1, p3t, l3t)
    host.flush()
    torch.cuda.synchronize()
    assert torch.equal(host.perm_d[1].cpu(), p3t) and torch.equal(host.lord_d[1].cpu(), l3t)
    assert int(env.stats[7].item()) == 0


def test_legal_count_and_emit_entry_points(D, oracle):
    """ddz_legal_count (closed form, no lists) == the list lengths; ddz_legal_emit == ddz_observe's packed lists."""
    B = 5000
    perm, lord = D.random_deals(B, seed=8)
    env = D.BatchedEnvComplicated(B, seed=6)
    env.prepare(perm, lord)
    for t in range(70):
        if t % 10 == 0:
            cnt = env.legal_counts()
            off = env.offsets.to(torch.int64)
            assert torch.equal(cnt.to(torch.int64), off[1:] - off[:-1])
        env.rollout_step()                                   # no re-deal: finished envs accumulate and count 0
    assert int((env.legal_counts() == 0).sum().item()) == int(env.is_done.sum().item()) > 0
    offs = torch.zeros(B + 1, dtype=torch.int32, device="cuda")
    acts = torch.zeros(env.cap, dtype=torch.int64, device="cuda")
    ws = torch.zeros(D.native.lib.ddz_workspace_bytes(B), dtype=torch.uint8, device="cuda")
    stats = torch.zeros(16, dtype=torch.int64, device="cuda")
    rc = D.native.lib.ddz_legal_emit(env._state.data_ptr(), ws.data_ptr(), offs.data_ptr(), acts.data_ptr(), env.cap,
                                     stats.data_ptr(), B, torch.cuda.current_stream().cuda_stream)
    assert rc == 0
    torch.cuda.synchronize()
    n = env.num_actions
    assert torch.equal(offs, env.offsets) and torch.equal(acts[:n], env.actions_packed) and int(stats[7].item()) == 0


def test_compressible_row_buffers(D):
    """ddz_rows_alloc / row_tensor: the face and one-hot buffers live in compressible device memory where the GPU has it;
    they behave like any other tensor, survive the allocator object going out of scope, and are given back on deletion."""
    import gc
    env = D.BatchedEnvCooperation(2048, seed=1)
    if not hasattr(env._face, "_ddz_rows"):
        pytest.skip("no compressible memory on this device / driver")
    perm, lord = D.random_deals(2048, seed=2)
    env.prepare(perm, lord)
    a = D.native.row_tensor((1000, 15, 4), "cuda")
    assert a.is_cuda and a.dtype == torch.float32 and a.shape == (1000, 15, 4) and a.data_ptr() % 256 == 0
    a.fill_(3.0)
    b = a.view(-1)[:60].clone()
    assert float(b.sum().item()) == 180.0
    free0 = torch.cuda.mem_get_info()[0]
    big = D.native.row_tensor((64 << 20,), "cuda")                   # 256 MB
    big.zero_()
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] <= free0 - (200 << 20)
    del big
    gc.collect()
    torch.cuda.synchronize()
    assert torch.cuda.mem_get_info()[0] >= free0 - (16 << 20)         # unmapped and released
    os.environ["DDZ_NO_COMPRESSION"] = "1"
    try:
        plain = D.BatchedEnvCooperation(2048, seed=1)
        assert not hasattr(plain._face, "_ddz_rows")
        plain.prepare(perm, lord)
        for _ in range(30):
            env.rollout_step(); plain.rollout_step()
        assert torch.equal(env.face, plain.face) and torch.equal(env.valid_actions()[0], plain.valid_actions()[0])
    finally:
        del os.environ["DDZ_NO_COMPRESSION"]


# ------------------------------------------------------------------ round 2: getters, multi-group host pipe, flat lists
def test_get_last_two_cards_batched_and_view(D, oracle, golden):
    """get_last_two_cards (envi.py:103-109; the rule bot reads it, rule_based/utils/rule_based_model.py:17-33): the batched
    getter against the oracle's envs every step (and its first non-empty entry against ddz_ref_env_last, the trick to
    beat), the B=1 view against the golden trace of the unmodified envi.py."""
    import ctypes as C
    B, G = 512, 2
    perm, lord = D.random_deals(B, seed=21, pool_games=G)
    env = D.BatchedEnvCooperation(B, seed=8)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env.prepare(pd, ld, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    L = oracle.lib()
    for t in range(90):
        got = env.get_last_two_cards().cpu().numpy()
        cur = ref.envs["cur"].astype(np.int64)
        rec = ref.envs["recent"]
        ar = np.arange(B)
        want = np.stack([rec[ar, (cur + 2) % 3], rec[ar, (cur + 1) % 3]], 1)
        assert np.array_equal(got, want), t
        for b in range(0, B, 37):                                # the trick to beat = first non-empty of the two
            last = np.zeros(15, np.int8)
            L.ddz_ref_env_last(C.c_void_p(ref.envs.ctypes.data + b * oracle.ENV_DTYPE.itemsize), last.ctypes.data_as(C.POINTER(C.c_int8)))
            first = got[b, 0] if got[b, 0].any() else got[b, 1]
            assert np.array_equal(first, last), (t, b)
        ref.observe(want_f32=False, want_face=False)
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=G)
        ref.step(mode=2, seed=8, env0=0, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=G)
    # B = 1 view: lists of card values like the reference's, replayed over the golden envi.py trace
    t = golden.envi_trace
    env1 = D.EnvCooperation()
    for g in range(3):
        env1.reset()
        env1.prepare(t["perms"][g][None], np.zeros(1, np.int8))
        prev = np.zeros((3, 15), np.int8)
        for s in np.flatnonzero(t["game"] == g):
            cur = int(t["role"][s])
            two = env1.get_last_two_cards()
            assert [list(map(int, x)) for x in two] == [list(D.Env.arr2cards(prev[(cur + 2) % 3])), list(D.Env.arr2cards(prev[(cur + 1) % 3]))]
            acts = env1.valid_actions()
            env1.step_manual(acts[int(t["choice"][s])])
            prev = t["recent"][s]


def test_host_rollout_groups_matches_oracle(D, oracle):
    """HostRolloutGroups: ONE native call per env-step of all groups of a GroupedEnv (ddz_mpipe_step) -- one H2D of the
    pinned entropy, one launch per group, one D2H of r/done/cat -- plus pool refills from the host.  Every step's results
    and the final state must equal the oracle's; all groups add to one shared stats vector."""
    B, P, NG = 2048, 2, 4
    rng = np.random.default_rng(77)
    perm, lord = D.random_deals(B, seed=19, pool_games=P)
    pool = [np.array(perm.reshape(P, B, 54)), np.array(lord.reshape(P, B))]
    ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=NG, seed=3)
    ge.prepare(perm, lord, pool_games=P)
    assert all(e.stats.data_ptr() == ge.stats.data_ptr() for e in ge.envs)
    host = D.HostRolloutGroups(ge)
    assert host.h2d_bytes == 4 * B and host.d2h_bytes == 3 * B
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=P)
    ents = [torch.as_tensor(rng.integers(0, 1 << 31, B).astype(np.int32)).pin_memory() for _ in range(5)]
    pending = []
    Bg = B // NG
    for t in range(130):
        if t % 40 == 20:
            slot = (t // 40) % P
            p2, l2 = D.random_deals(B, seed=500 + t)
            host.refill(slot, torch.as_tensor(p2).pin_memory(), torch.as_tensor(l2).pin_memory(), now=(t != 60))
            if t == 60:
                host.flush()
            pool[0][slot], pool[1][slot] = p2, l2
        res = host.step(ents[t % 5])
        ref.observe(want_f32=False, want_face=False)
        rr, rd, rc, _ = ref.step(ents[t % 5].numpy(), mode=1)
        ref.deal(pool[0].reshape(-1, 54), pool[1].reshape(-1), only_done=True, pool_games=P)
        pending.append((res, rr.copy(), rd.copy(), rc.copy(), t))
        if len(pending) == 3:                         # read two steps late, as a pipelined host would
            got, rr, rd, rc, tt = pending.pop(0)
            D.HostRolloutGroups.wait(got)
            for g in range(NG):
                sl = slice(g * Bg, (g + 1) * Bg)
                assert np.array_equal(got.r[g], rr[sl]) and np.array_equal(got.done[g], rd[sl]) and np.array_equal(got.cat[g], rc[sl]), (tt, g)
    ge.join()
    torch.cuda.synchronize()
    f, meta = ref.export()
    got_f = torch.cat([e._fields()[0] for e in ge.envs], 1).cpu().numpy().view(np.uint64)
    got_m = torch.cat([e._fields()[1] for e in ge.envs]).cpu().numpy().view(np.uint32)
    assert np.array_equal(got_f, f) and np.array_equal(got_m, meta)
    st = ge.stats.cpu().numpy()
    assert st[7] == 0 and st[4] == ref.stats[4] == 130 * B and st[0] == ref.stats[0] > 0
    for g, e in enumerate(ge.envs):                   # the lists after the last step are those of the final state
        off = e.offsets.cpu().numpy()
        sub = oracle.RefBatch(Bg, 2)
        sub.envs[:] = ref.envs[g * Bg:(g + 1) * Bg]
        want_off, want_au, _, want_face = sub.observe(want_f32=False)
        assert np.array_equal(off, want_off) and np.array_equal(e.actions_packed.cpu().numpy().view(np.uint64), want_au)
        assert np.array_equal(e.face.cpu().numpy(), want_face)


def test_legal_moves_multi_round_tiles_and_long_lists(D, oracle):
    """ddz_legal_moves (k_legal_flat) on tiles made only of the heaviest hands: several arena rounds per tile, windows that
    straddle hands and rounds, an odd list base, plus a tile of tiny hands behind them."""
    rng = np.random.default_rng(3)
    heavy = D.ADVERSARIAL_POOL[[0, 1, 3, 8, 9]]
    hands = np.concatenate([heavy[rng.integers(0, len(heavy), 75)], _rand_hands(rng, 40, 1, 4), heavy[rng.integers(0, len(heavy), 45)]])
    n = len(hands)
    z = np.zeros(15, np.int8)
    lasts = np.zeros((n, 15), np.int8)
    lasts[0] = np.eye(15, dtype=np.int8)[2]               # an odd number of moves in front of everything else
    for i in range(1, n, 3):
        om = oracle.get_moves(heavy[rng.integers(0, len(heavy))], z, fast=True)
        lasts[i] = om[rng.integers(0, len(om))]
    packed, offsets = D.get_moves(hands, lasts)
    for i, got in enumerate(_split(packed, offsets)):
        want = oracle.pack(oracle.get_moves(hands[i], lasts[i], fast=True))
        assert np.array_equal(got, np.atleast_1d(want)), (i, hands[i], lasts[i])


def test_prob_form_b_build_matches_form_b_oracle(D):
    """The build switch for the one layout nothing in the reference pins (oracle/SEMANTICS.md, server/core.py:26-33): the
    library and the oracle compiled with -DDDZ_PROB_FORM_B agree bit for bit on all four faces (the default build, form A,
    is what every other test checks)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_b = os.path.join(root, "doudizhu-rl_b200", "libddz_b200_formB.so")
    ora_b = os.path.join(root, "oracle", "libddz_oracle_formB.so")
    if not (os.path.exists(lib_b) and os.path.exists(ora_b)):
        import __graft_entry__
        __graft_entry__.build()
    assert D.native.lib.ddz_prob_form() == 0
    env = dict(os.environ, DDZ_LIB=lib_b, DDZ_ORACLE_LIB=ora_b)
    out = subprocess.run([sys.executable, os.path.join(root, "tests", "form_b_check.py")], env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "form B ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def test_uct_search_equals_reference_algorithm_on_oracle(D, oracle):
    """The search bot (server/mcts/interface.py:37-45): UctSearch (tree on the host, legal moves and playouts on the device)
    against the reference algorithm restated over the oracle (tests/uct_reference_algorithm.py), same seed and budget:
    the same tree statistics at the root and the same chosen move, for the sequential search (width 1) and a wide one,
    over the full move lists and over the bot's pruned ones (the reference's own configuration)."""
    from uct_reference_algorithm import uct
    z = np.zeros((3, 15), np.int64)
    positions = []
    h = np.zeros((3, 15), np.int64); h[1, [0, 1, 2, 3, 4, 9]] = [1, 1, 1, 1, 1, 2]; h[2, [5, 6]] = 2; h[0, [10, 11, 12]] = [1, 2, 1]
    positions.append((1, h, z))                                       # the landlord leads
    h2 = np.zeros((3, 15), np.int64); h2[2, [7, 7 + 1, 12]] = [2, 1, 1]; h2[0, [0, 3]] = [1, 2]; h2[1, [1, 5, 13]] = [1, 1, 1]
    last = z.copy(); last[1, 6] = 2                                   # down must beat the landlord's pair of 9s (or pass)
    positions.append((2, h2, last))
    rng = np.random.default_rng(4)
    deck = np.array([i // 4 for i in range(52)] + [13, 14])
    p = rng.permutation(deck)[:21]
    h3 = np.stack([np.bincount(p[0:7], minlength=15), np.bincount(p[7:15], minlength=15), np.bincount(p[15:21], minlength=15)]).astype(np.int64)
    positions.append((0, h3, z))
    p = rng.permutation(deck)[:45]                                    # mid-game hands: lists long enough to be pruned
    h4 = np.stack([np.bincount(p[0:14], minlength=15), np.bincount(p[14:31], minlength=15), np.bincount(p[31:45], minlength=15)]).astype(np.int64)
    positions.append((1, h4, z))
    assert len(oracle.get_moves(h4[1], z[0], fast=True)) > 10
    for k, (role, hands, last) in enumerate(positions):
        for width, budget, prune in ((1, 120, False), (16, 60, False), (1, 100, True), (8, 50, True)):
            want_move, want_root = uct(oracle, role, hands, last, budget, width=width, seed=7 + k, prune=prune)
            s = D.UctSearch(role, hands, last, width=width, seed=7 + k, prune=prune).run(budget)
            moves, visits, rate = s.root_table()
            assert len(moves) == len(want_root.children), (k, width)
            for i, ch in enumerate(want_root.children):
                assert np.array_equal(moves[i], ch.state.action) and visits[i] == ch.visit and rate[i] == ch.reward / ch.visit, (k, width, i)
            assert np.array_equal(s.best_move(), want_move), (k, width)
            assert s.playouts <= budget * width and s.iterations == budget


def test_host_rollout_groups_chunked_deferred_refill(D):
    """HostRolloutGroups.refill: the upload goes up in 384 KB chunks, one per step; every group's slot is replaced whole,
    between two of its steps, by the first step that finds the upload complete -- never a mixture of old and new rows."""
    B, P, NG = 32768, 2, 4                                    # 1.7 MB of permutations: five chunks
    perm, lord = D.random_deals(B, seed=1, pool_games=P)
    ge = D.GroupedEnv(D.BatchedEnvCooperation, B, groups=NG, seed=3, max_actions_per_env=160)
    ge.prepare(perm, lord, pool_games=P)
    host = D.HostRolloutGroups(ge)
    ent = torch.as_tensor(np.random.default_rng(0).integers(0, 1 << 31, B).astype(np.int32)).pin_memory()
    p2, l2 = D.random_deals(B, seed=77)
    p2t, l2t = torch.as_tensor(p2).pin_memory(), torch.as_tensor(l2).pin_memory()
    Bg = B // NG
    old = [ge._pool[g][0][1].clone().cpu() for g in range(NG)]
    host.refill(1, p2t, l2t)
    replaced_at = None
    for t in range(200):
        res = host.step(ent)
        ge.join(); torch.cuda.synchronize()
        state = []
        for g in range(NG):
            slot = ge._pool[g][0][1].cpu()
            new = p2t[g * Bg:(g + 1) * Bg]
            assert torch.equal(slot, old[g]) or torch.equal(slot, new), (t, g)      # never a mixture
            state.append(torch.equal(slot, new))
        if all(state):
            replaced_at = t
            break
    assert replaced_at is not None and replaced_at >= 3          # the chunks take a few steps
    D.HostRolloutGroups.wait(res)
    for g in range(NG):
        assert torch.equal(ge._pool[g][1][1].cpu(), l2t[g * Bg:(g + 1) * Bg])
    assert int(ge.stats[7].item()) == 0


def test_config3_parity_at_full_size_with_the_256_wide_net(D, oracle):
    """BASELINE config 3 at its own size: 65 536 envs, the landlord = argmax Q with a network of NetCooperation's layer
    sizes (10 x 15 x 4 in, 256-wide convolutions, 256 hidden; net.py:125-139), farmers random, 24 steps.  Every step the
    GPU env's offsets / packed lists / face equal the oracle's; the Q-values that the in-place [n, C+1, 15, 4] encoder + the
    network give equal those of the reference formulation (face.repeat + torch.cat, net.py:87-90) on a sample of envs, and
    so do the argmax decisions; both envs then take the same decisions and end in the same state."""
    from qnet_like import QNetLike
    torch.manual_seed(0)
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False     # fp32 network, as in the reference
    B, G, steps = 65536, 2, 24
    net = QNetLike(9, width=256, hidden=256).cuda().eval()
    policy = D.BatchedGreedyPolicy(net, chunk_actions=1 << 16)
    perm, lord = D.random_deals(B, seed=23, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    prev = D.native.set_tile_order("ticket")                       # the network's kernels share the GPU with the env launches
    try:
        env = D.BatchedEnvCooperation(B, max_actions_per_env=160)
        env.prepare(pd, ld, pool_games=G)
        ref = oracle.RefBatch(B, 2)
        ref.deal(perm, lord, pool_games=G)
        gen = torch.Generator(device="cuda"); gen.manual_seed(5)
        sample = torch.arange(0, B, 53, device="cuda")[:1024]
        for t in range(steps):
            o_off, o_au, _, o_face = ref.observe(want_f32=False)
            off = env.offsets
            assert np.array_equal(off.cpu().numpy(), o_off), t
            assert np.array_equal(env.actions_packed.cpu().numpy().view(np.uint64), o_au), t
            assert np.array_equal(env.face.cpu().numpy(), o_face), t
            is_lord = env.get_role_ID() == 2
            q = policy.q_values(env, is_lord)
            greedy = policy.select(env, q)
            # the reference formulation on a sample of the landlord's envs
            acts, _ = env.valid_actions()
            offc = off.cpu().numpy()
            with torch.no_grad():
                for b in sample[is_lord[sample]].tolist()[:96]:
                    lo, hi = int(offc[b]), int(offc[b + 1])
                    want = net(env.face[b], acts[lo:hi]).reshape(-1)
                    # fp32 either way, but other batch shapes pick other convolution / GEMM algorithms: tolerance 1e-3 relative
                    assert torch.allclose(q[lo:hi], want, rtol=1e-3, atol=1e-4), (t, b, (q[lo:hi] - want).abs().max().item())
                    assert int(greedy[b]) == int(torch.argmax(q[lo:hi]))
            cnt = off[1:] - off[:-1]
            ent = torch.randint(0, 1 << 30, (B,), device="cuda", dtype=torch.int32, generator=gen)
            choice = torch.where(is_lord, greedy, ent % cnt.clamp(min=1)).to(torch.int32)
            env.rollout_step(choice, mode=D.native.CHOICE_INDEX, perm=pd, lord_pile=ld, pool_games=G)
            ref.step(choice.cpu().numpy(), mode=0)
            ref.deal(perm, lord, only_done=True, pool_games=G)
        _compare_state(env, ref, steps)
        st = env.stats.cpu().numpy()
        assert st[7] == 0 and np.array_equal(st[[0, 1, 2, 3, 4]], ref.stats[[0, 1, 2, 3, 4]]) and st[4] == B * steps
    finally:
        D.native.set_tile_order(prev)
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32


def test_legal_moves_respect_the_list_capacity(D, oracle):
    """ddz_legal_moves with a buffer smaller than the lists: the stored prefix is exact, nothing is written past `cap`
    (odd and even caps: the kernel stores pairs of moves), the offsets are those of the complete lists, stats[7] says so."""
    rng = np.random.default_rng(8)
    hands = np.concatenate([D.ADVERSARIAL_POOL[rng.integers(0, 10, 40)], _rand_hands(rng, 60, 5, 21)]).astype(np.int8)
    lasts = np.zeros_like(hands)
    want = [np.atleast_1d(oracle.pack(oracle.get_moves(h, l, fast=True))) for h, l in zip(hands, lasts)]
    flat = np.concatenate(want)
    hp = D.pack_counts(torch.as_tensor(hands).cuda()).contiguous()
    lp = torch.zeros(len(hands), dtype=torch.int64, device="cuda")
    for cap in (len(flat) + 5, len(flat), len(flat) - 1, 1001, 1000, 7, 0):
        gen = D.MoveGenerator(len(hands), max_moves_per_hand=1)
        gen.cap = cap
        gen.actions = torch.full((len(flat) + 64,), -1, dtype=torch.int64, device="cuda")
        acts, offs = gen.generate(hp, lp)
        torch.cuda.synchronize()
        got = acts.cpu().numpy()
        keep = min(cap, len(flat))
        assert np.array_equal(got[:keep].view(np.uint64), flat[:keep]), cap
        assert (got[keep:] == -1).all(), cap
        assert np.array_equal(offs.cpu().numpy(), np.concatenate([[0], np.cumsum([len(w) for w in want])])), cap
        assert int(gen.stats[7].item()) == (1 if cap < len(flat) else 0), cap


def test_graph_replay_after_steps_that_bypass_the_device_counter(D, oracle):
    """Only the fused launches keep the device-side Philox step counter up to date.  step_random() (ddz_step) and a state
    restored with load_state_dict advance / set the step number on the host alone: a graph replay after them must re-arm
    the counter, or it would draw moves from step numbers that were already used."""
    B, G, seed = 512, 4, 77
    perm, lord = D.random_deals(B, seed=2, pool_games=G)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = D.BatchedEnvCooperation(B, seed=seed)
    env.prepare(pd, ld, pool_games=G)
    ref = oracle.RefBatch(B, 2)
    ref.deal(perm, lord, pool_games=G)
    t = 0

    def ref_steps(k):
        nonlocal t
        for _ in range(k):
            ref.observe(want_f32=False, want_face=False)
            ref.step(mode=2, seed=seed, step=t); ref.deal(perm, lord, only_done=True, pool_games=G); t += 1

    gr = D.GraphedRollout(env, pd, ld, G)
    for _ in range(5):
        gr.replay()
    ref_steps(10)
    for _ in range(3):                                   # eager steps through ddz_step: the device counter does not see them
        env.step_random()
        env.prepare(pd, ld, only_done=True, pool_games=G)
    ref_steps(3)
    for _ in range(4):
        gr.replay()
    ref_steps(8)
    _compare_state(env, ref, t)
    sd = env.state_dict()
    for _ in range(3):
        gr.replay()
    env.load_state_dict(sd)                              # back to step 21: the counter must follow
    for _ in range(2):
        gr.replay()
    ref_steps(4)
    _compare_state(env, ref, t)
    _compare_observation(env, ref, t)
    assert int(env.stats[7].item()) == 0


def test_bench_dump_outputs_are_reproducible(D, oracle, tmp_path):
    """bench.py --dump-outputs: two runs with the same arguments write the same arrays (float32 / float64, a fixed sample
    of the envs), and they are what the last timed step returned: the oracle, replaying the bench's deals and Philox
    streams for prefill + warm-up + timed steps, gives the same r / done / cat / reward of that step and the same face
    and legal lists of the state after it, env by env."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    import bench
    B, steps = 12288, 3                                  # more envs than the dump samples
    dumps = []
    for run in range(2):
        out_dir = str(tmp_path / ("run%d" % run))
        cmd = [sys.executable, os.path.join(root, "bench.py"), "--envs", str(B), "--steps", str(steps), "--warmup", "2",
               "--prefill", "20", "--no-cpu-baseline", "--no-single", "--clock-interval-ms", "0", "--dump-outputs", out_dir]
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["verify"] == "ok"
        dumps.append({f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))})
    a, b = dumps
    assert sorted(a) == ["cat", "done", "env_index", "face", "legal_actions", "legal_counts", "r", "reward"]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for name in a:
        assert a[name].dtype in (np.float32, np.float64) and np.array_equal(a[name], b[name]), name
    idx = a["env_index"].astype(np.int64)
    assert len(idx) == bench.DUMP_ENVS and (np.diff(idx) > 0).all() and idx[-1] < B
    assert a["legal_actions"].shape == (int(a["legal_counts"].sum()), 15, 4)

    P, seed = bench.POOL_GAMES, bench.SEED
    perm, lord = D.random_deals(B, seed=seed, pool_games=P)
    ref = oracle.RefBatch(B, variant=bench.VARIANT)
    ref.deal(perm, lord, pool_games=P)
    for t in range(line["config"]["prefill_steps"] + line["config"]["warmup_env_steps"] + steps):
        ref.observe(want_f32=False, want_face=False)
        r, done, cat, rew = ref.step(mode=2, seed=seed, env0=0, step=t)
        ref.deal(perm, lord, only_done=True, pool_games=P)
    off, _, af, face = ref.observe()
    for name, want in (("r", r), ("done", done), ("cat", cat), ("reward", rew), ("face", face), ("legal_counts", np.diff(off))):
        assert np.array_equal(a[name], want[idx].astype(np.float32)), name
    assert np.array_equal(a["legal_actions"], np.concatenate([af[off[i]:off[i + 1]] for i in idx]))
