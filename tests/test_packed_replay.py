"""Packed replay: ddz_encode_face_gather (csrc/ddz_kernels.cu, k_face_gather), trainer.PackedReplayBuffer,
TransitionCollector(packed=True) and BatchedGame(replay="packed").

The kernel's reference is the library's own face and action encoders over the same rows: ddz_encode_face over the gathered
state and ddz_encode_actions over the gathered moves (both pinned to the oracle elsewhere), and for the concatenated layout
the rows of env.state_actions().  The packed path as a whole is checked against the float path: the golden transitions of
the unmodified game.py, and a float and a packed BatchedGame that play the same games."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

SENTINEL = 0x7FBADBAD                     # a NaN bit pattern no kernel writes
CLASSES = [("BatchedEnv", 4), ("BatchedEnvComplicated", 7), ("BatchedEnvCooperation", 9), ("BatchedEnvCooperationSimplify", 6)]
SIZES = [0, 1, 31, 32, 33, 4097]


def _lib():
    import ddz_b200 as D
    return D.native


# ------------------------------------------------------------------------------------------------ CPU
def test_face_gather_argument_checks():
    """every bad argument is refused before any CUDA call (so this runs without a GPU)"""
    N = _lib()
    L, E, S, K = N.lib, N.E_ARG, N.ROWS_SPLIT, N.ROWS_CONCAT
    # (state, variant, rows, n, moves, face, move_rows, layout, B)
    bad = [
        (None, 0, 1, 4, 1, 1, None, S, 8),          # NULL state with n > 0
        (1, 0, None, 4, 1, 1, None, S, 8),          # NULL rows
        (1, 0, 1, 4, 1, None, None, S, 8),          # NULL face
        (1, 0, 1, -1, 1, 1, None, S, 8),            # n < 0
        (1, 0, 1, 4, 1, 1, None, S, 0),             # B <= 0
        (1, 0, 1, 4, 1, 1, None, S, -3),
        (1, 4, 1, 4, 1, 1, None, S, 8),             # unknown variant
        (1, -1, 1, 4, 1, 1, None, S, 8),
        (1, 0, 1, 4, 1, 1, None, 2, 8),             # unknown layout
        (1, 0, 1, 4, 1, 1, None, -1, 8),
        (1, 0, 1, 4, None, 1, None, K, 8),          # CONCAT without moves
        (1, 0, 1, 0, None, 1, None, K, 8),          # ... also with n = 0
        (1, 0, 1, 4, None, 1, 1, S, 8),             # SPLIT with move_rows but no moves
        (1, 0, 1, 4, 1, 1, 1, K, 8),                # move_rows with CONCAT
        (None, 0, None, 0, None, None, None, S, 0),  # n = 0 does not excuse B <= 0
    ]
    for args in bad:
        assert L.ddz_encode_face_gather(*args, None) == E, args
    # n = 0: nothing to do, no launch (so 0 even without a device), NULL buffers allowed
    assert L.ddz_encode_face_gather(None, 2, None, 0, None, None, None, S, 8, None) == 0
    assert L.ddz_encode_face_gather(None, 3, None, 0, 1, None, None, K, 8, None) == 0


def _labelled(n, base, channels=2):
    """n float transitions and the packed transitions carrying the same labels (base + i)"""
    import ddz_b200 as D
    lab = torch.arange(base, base + n, dtype=torch.int64)
    fl = (lab.float()[:, None, None, None].expand(n, channels, 15, 4).clone(), lab.float()[:, None, None].expand(n, 15, 4).clone(),
          lab.float(), (lab.float() + 0.5)[:, None, None, None].expand(n, channels, 15, 4).clone(),
          (lab.float() + 0.5)[:, None, None].expand(n, 15, 4).clone(), (lab % 2).float())
    s0 = torch.zeros(D.native.STATE_WORDS * n, dtype=torch.int32)
    s1 = torch.zeros_like(s0)
    for s, off in ((s0, 0), (s1, 1000000)):
        f, meta = D.trainer.state_fields(s, n)
        f.copy_((lab + off)[None, :].expand(9, n) * torch.arange(1, 10)[:, None])
        meta.copy_((lab + off).to(torch.int32))
    pk = (s0, lab * 16, lab.float(), s1, lab * 16 + 1, (lab % 2).float())
    return fl, pk


def test_packed_ring_bookkeeping_matches_replay_buffer():
    """PackedReplayBuffer's ring == ReplayBuffer's (head, size, the slot of every transition): wrap-around, a batch larger
    than the capacity, capacity 1 and empty appends, on CPU tensors"""
    import ddz_b200 as D
    for cap, sizes in ((7, [3, 0, 4, 5, 0, 13, 2, 7, 1]), (1, [1, 0, 3, 1, 2]), (5, [5, 5, 6, 0, 4, 11])):
        rb = D.ReplayBuffer(cap, 2, "cpu")
        pb = D.PackedReplayBuffer(cap, D.native.FACE_FIRST, "cpu")
        base = 1
        for n in sizes:
            fl, pk = _labelled(n, base)
            base += n
            rb.append(*fl)
            pb.append(*pk)
            assert (pb.head, pb.size, len(pb)) == (rb.head, rb.size, len(rb)), (cap, n)
            assert torch.equal(pb.r, rb.r) and torch.equal(pb.done, rb.done), (cap, n)
            lab = rb.r[:, 0].to(torch.int64)                       # the label of every slot (0 = never written)
            f, meta = D.trainer.state_fields(pb.state, 2 * cap)
            filled = lab > 0
            assert torch.equal(rb.s0[:, 0, 0, 0].to(torch.int64), lab) and torch.equal(rb.s1[:, 0, 0, 0], rb.r[:, 0] + 0.5 * filled)
            assert torch.equal(meta[:cap].to(torch.int64), lab)
            assert torch.equal(meta[cap:].to(torch.int64), (lab + 1000000) * filled)
            assert torch.equal(f[:, :cap], lab[None, :] * torch.arange(1, 10)[:, None])
            assert torch.equal(f[:, cap:], ((lab + 1000000) * filled)[None, :] * torch.arange(1, 10)[:, None])
            assert torch.equal(pb.moves[:cap], lab * 16) and torch.equal(pb.moves[cap:], (lab * 16 + 1) * filled)
    assert D.PackedReplayBuffer.bytes_per_transition == 176
    with pytest.raises(ValueError):
        D.PackedReplayBuffer(4, 7, "cpu")


# ------------------------------------------------------------------------------------------------ GPU helpers
@pytest.fixture(scope="module")
def D():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    import ddz_b200
    return ddz_b200


def fresh_env(D, cls, B, seed=1):
    env = getattr(D, cls)(B, seed=seed)
    perm, lord = D.random_deals(B, seed=seed + B)
    env.prepare(perm, lord)
    return env


def midgame_env(D, cls, B=4096, steps=23, seed=3):
    """re-dealt as games end: positions at every depth"""
    perm, lord = D.random_deals(B, seed=seed, pool_games=2)
    pd, ld = torch.as_tensor(perm).cuda(), torch.as_tensor(lord).cuda()
    env = getattr(D, cls)(B, seed=seed)
    env.prepare(pd, ld, pool_games=2)
    for _ in range(steps):
        env.rollout_step(perm=pd, lord_pile=ld, pool_games=2)
    return env


def finished_env(D, cls, B=4096, steps=40, seed=4):
    """no re-deal: some envs are finished"""
    env = fresh_env(D, cls, B, seed)
    for _ in range(steps):
        env.rollout_step()
    assert 0 < int(env.is_done.sum()) < B
    return env


def payload_env(D, cls, golden):
    """the core payloads (placeholder hands for the two players the payload does not show)"""
    g = golden.core_payloads
    return D.env_from_arrays(g["role"], g["hand"], g["history"], g["last_taken"], g["left"], env_cls=getattr(D, cls))


def env_moves(env, rng):
    """one packed move per env: a legal one, a pass (0) or an arbitrary 64-bit pattern (the one-hot is defined for any)"""
    B = env.B
    off = env.offsets.to(torch.int64)
    cnt = off[1:] - off[:-1]
    au = env.actions_packed
    pick = torch.as_tensor(rng.integers(0, 1 << 30, B), device="cuda") % cnt.clamp(min=1)
    legal = au[(off[:-1] + pick).clamp(max=max(au.numel() - 1, 0))] * (cnt > 0) if au.numel() else torch.zeros(B, dtype=torch.int64, device="cuda")
    junk = torch.as_tensor(rng.integers(-(1 << 63), (1 << 63) - 1, B, dtype=np.int64), device="cuda")
    kind = torch.as_tensor(rng.integers(0, 4, B), device="cuda")
    return torch.where(kind == 0, torch.zeros_like(junk), torch.where(kind == 1, junk, legal)).contiguous()


def sample_rows(rng, B, n):
    """rows with duplicates, a reversed run and rows outside [0, B)"""
    rows = rng.integers(-3, B + 3, n)
    if n > 8:
        rows[: n // 4] = np.arange(n // 4)[::-1] % B
        rows[n // 4: n // 4 + 4] = [-1, B, B + 1000, -(1 << 40)]
    return torch.as_tensor(rows, dtype=torch.int64, device="cuda")


def gather(D, state, B, variant, rows, moves, layout, with_moves=True, guard=64):
    """the launch through the C-ABI into sentinel-filled buffers; checks that the guard rows after the output stay untouched"""
    N = D.native
    C = N.lib.ddz_face_channels(variant)
    n = rows.numel()
    R = C + 1 if layout == N.ROWS_CONCAT else C
    face = torch.full(((n + guard) * R * 60,), SENTINEL, dtype=torch.int32, device="cuda")
    mv = torch.full(((n + guard) * 60,), SENTINEL, dtype=torch.int32, device="cuda") if with_moves and layout == N.ROWS_SPLIT else None
    rc = N.lib.ddz_encode_face_gather(state.data_ptr(), variant, rows.data_ptr(), n, moves.data_ptr() if moves is not None else None,
                                      face.data_ptr(), mv.data_ptr() if mv is not None else None, layout, B,
                                      torch.cuda.current_stream().cuda_stream)
    N.check(rc, "ddz_encode_face_gather")
    assert bool((face[n * R * 60:] == SENTINEL).all()), "face guard overwritten"
    out_face = face[: n * R * 60].view(torch.float32).view(n, R, 15, 4)
    if mv is None:
        return out_face, None
    assert bool((mv[n * 60:] == SENTINEL).all()), "move-row guard overwritten"
    return out_face, mv[: n * 60].view(torch.float32).view(n, 15, 4)


def encode_face(D, state, variant, B):
    C = D.native.lib.ddz_face_channels(variant)
    face = torch.empty((B, C, 15, 4), dtype=torch.float32, device="cuda")
    D.native.check(D.native.lib.ddz_encode_face(state.data_ptr(), variant, face.data_ptr(), B,
                                                torch.cuda.current_stream().cuda_stream), "ddz_encode_face")
    return face


def reference(D, env, rows, moves):
    """ddz_encode_face over the gathered state + ddz_encode_actions over the gathered moves; zero rows for rows outside [0, B)"""
    ok = (rows >= 0) & (rows < env.B)
    safe = torch.where(ok, rows, torch.zeros_like(rows))
    n = rows.numel()
    if n == 0:
        return (torch.zeros((0, env.C, 15, 4), device="cuda"), torch.zeros((0, 15, 4), device="cuda"))
    face = encode_face(D, D.gather_states(env, safe), env.VARIANT, n) * ok[:, None, None, None]
    acts = env.encode_actions(moves[safe] * ok)
    return face, acts


def check_gather(D, env, rng, sizes):
    """SPLIT with and without move rows and CONCAT against the reference, bit for bit, for every n in sizes"""
    N, B, V = D.native, env.B, env.VARIANT
    moves = env_moves(env, rng)
    for n in sizes:
        rows = sample_rows(rng, B, n)
        want_face, want_mv = reference(D, env, rows, moves)
        face, mv = gather(D, env._state, B, V, rows, moves, N.ROWS_SPLIT)
        assert torch.equal(face.view(torch.int32), want_face.view(torch.int32)), (type(env).__name__, B, n)
        assert torch.equal(mv.view(torch.int32), want_mv.view(torch.int32)), (type(env).__name__, B, n)
        face2, none = gather(D, env._state, B, V, rows, None, N.ROWS_SPLIT, with_moves=False)
        assert none is None and torch.equal(face2.view(torch.int32), want_face.view(torch.int32))
        cat, _ = gather(D, env._state, B, V, rows, moves, N.ROWS_CONCAT)
        assert torch.equal(cat.view(torch.int32), torch.cat((want_face, want_mv[:, None]), 1).view(torch.int32)), (B, n)


# ------------------------------------------------------------------------------------------------ GPU: the kernel
@pytest.mark.gpu
@pytest.mark.parametrize("cls,C", CLASSES)
def test_gather_equals_face_and_action_encoders(D, golden, cls, C):
    rng = np.random.default_rng(C)
    for B in (1, 7, 4096):
        check_gather(D, fresh_env(D, cls, B), rng, SIZES)
    mid = midgame_env(D, cls)
    check_gather(D, mid, rng, SIZES + [1 << 20])
    check_gather(D, finished_env(D, cls), rng, SIZES)
    check_gather(D, payload_env(D, cls, golden), rng, SIZES)


@pytest.mark.gpu
@pytest.mark.parametrize("cls,C", CLASSES)
def test_concat_rows_equal_state_actions(D, golden, cls, C):
    """DDZ_ROWS_CONCAT with rows = the owner env of every legal move and moves = that move: env.state_actions() row for row"""
    for env in (midgame_env(D, cls, B=2000), finished_env(D, cls, B=600), payload_env(D, cls, golden)):
        off = env.offsets.to(torch.int64)
        cnt = off[1:] - off[:-1]
        au = env.actions_packed
        want = env.state_actions()[0]
        got = torch.empty_like(want)
        # one launch per move index j: env b's move j goes to row off[b] + j (moves is indexed by env)
        for j in range(int(cnt.max())):
            has = cnt > j
            moves = torch.where(has, au[(off[:-1] + j).clamp(max=au.numel() - 1)], torch.zeros_like(off[:-1]))
            rows = torch.arange(env.B, device="cuda")[has]
            x = D.decode_rows(env._state, env.VARIANT, rows, moves, concat=True)
            got[off[:-1][has] + j] = x
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), cls


@pytest.mark.gpu
def test_form_b_build_gather():
    """the gather against ddz_encode_face of the -DDDZ_PROB_FORM_B build, all four variants, in a subprocess"""
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    lib_b = os.path.join(root, "doudizhu-rl_b200", "libddz_b200_formB.so")
    if not os.path.exists(lib_b):
        import __graft_entry__
        __graft_entry__.build()
    out = subprocess.run([sys.executable, os.path.join(root, "tests", "form_b_replay_check.py")],
                         env=dict(os.environ, DDZ_LIB=lib_b), capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "form B replay ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


# ------------------------------------------------------------------------------------------------ GPU: collector and buffers
@pytest.mark.gpu
def test_packed_collector_matches_reference_game_loop(D, oracle, golden):
    """the 40-deal recorded-index run of test_transition_assembly_matches_reference_game_loop with packed=True: decoding
    every emitted transition gives the (s0, a0, r, s1, a1, done) the UNMODIFIED game.py's perceive() received"""
    g = golden.game_transitions
    seed, perms = int(g["seed"]), g["perms"]
    B = len(perms)
    env = D.BatchedEnvCooperation(B, debug=True)
    env.prepare(perms, np.zeros(B, np.int8))
    col = D.TransitionCollector(env, role=1, reward=100.0, packed=True)
    got = [[] for _ in range(B)]

    def take(out):
        s0, a0, r, s1, a1, done, idx = out
        n = idx.numel()
        assert s0.dtype == torch.int32 and s0.numel() == 19 * n and a0.dtype == torch.int64 and a0.shape == (n,)
        rows = torch.arange(n, device="cuda")
        f0, m0 = D.decode_rows(s0, env.VARIANT, rows, a0) if n else (torch.zeros(0, 9, 15, 4), torch.zeros(0, 15, 4))
        f1, m1 = D.decode_rows(s1, env.VARIANT, rows, a1) if n else (f0, m0)
        f0, m0, r, f1, m1, done, idx = (x.cpu().numpy() for x in (f0, m0, r, f1, m1, done, idx))
        for i, b in enumerate(idx):
            got[b].append((f0[i], m0[i], float(r[i]), f1[i], m1[i], bool(done[i])))

    for t in range(200):
        acts, offs = env.valid_actions()
        au = env.actions_packed
        off = offs.cpu().numpy().astype(np.int64)
        cnt = np.diff(off)
        k0 = np.array([oracle.philox(seed, b, 2 * t) % cnt[b] if cnt[b] else 0 for b in range(B)])
        k1 = np.array([oracle.philox(seed, b, 2 * t + 1) % cnt[b] if cnt[b] else 0 for b in range(B)])
        live = torch.as_tensor(cnt > 0).cuda()
        a0 = au[torch.as_tensor(np.minimum(off[:-1] + k0, max(off[-1] - 1, 0))).cuda()] * live
        a1 = au[torch.as_tensor(np.minimum(off[:-1] + k1, max(off[-1] - 1, 0))).cuda()] * live
        take(col.on_turn(a0, a1))
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


def _game(D, cls, C, replay, B=256, **kw):
    from qnet_like import QNetLike
    net = lambda: QNetLike(C, width=16, seed=11)          # every construction has the same weights
    return D.BatchedGame(getattr(D, cls), {"lord": net, "down": net, "up": None},
                         {"lord": D.BatchedDQN, "down": D.BatchedDQN, "up": None}, reward_dict={"lord": 100, "down": 50, "up": 50},
                         train_dict={"lord": True, "down": True, "up": False}, seed=9, num_envs=B, replay=replay, **kw)


def _bits(x):
    return x.contiguous().view(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("cls,C", CLASSES)
def test_float_and_packed_buffers_hold_the_same_data(D, cls, C):
    """two BatchedGames, same seed, frozen nets (updates_per_step=0): identical games, so the packed buffer decodes to the
    float buffer slot for slot, sample() with cloned generators is bit-identical, and a TD step gives the same loss"""
    gf = _game(D, cls, C, "float", updates_per_step=0)
    gp = _game(D, cls, C, "packed", updates_per_step=0)
    assert isinstance(gf.lord.replay_buffer, D.ReplayBuffer) and isinstance(gp.lord.replay_buffer, D.PackedReplayBuffer)
    assert not gf._collectors["lord"].packed and gp._collectors["lord"].packed
    for _ in range(300):
        gf.step()
        gp.step()
    assert torch.equal(gf.env._state, gp.env._state) and gf.episodes == gp.episodes > 0
    for role in ("lord", "down"):
        rb, pb = getattr(gf, role).replay_buffer, getattr(gp, role).replay_buffer
        assert (rb.size, rb.head) == (pb.size, pb.head) and rb.size > 4096
        idx = torch.arange(rb.size, device="cuda")
        for want, got in zip((rb.s0, rb.a0, rb.r, rb.s1, rb.a1, rb.done), pb.decode(idx)):
            assert torch.equal(_bits(got), _bits(want[idx])), role
        g1, g2 = torch.Generator(device="cuda"), torch.Generator(device="cuda")
        g1.manual_seed(5)
        g2.set_state(g1.get_state())
        for want, got in zip(rb.sample(4096, g1), pb.sample(4096, g2)):
            assert torch.equal(_bits(got), _bits(want)), role
    # one TD step on each from identical nets and optimizer states
    af, ap = gf.lord, gp.lord
    ap.policy_net.load_state_dict(af.policy_net.state_dict())
    ap.target_net.load_state_dict(af.target_net.state_dict())
    ap.optimizer.load_state_dict(af.optimizer.state_dict())
    af._gen.manual_seed(77)
    ap._gen.manual_seed(77)
    lf = D.td_step(af.policy_net, af.target_net, af.optimizer, af.replay_buffer.sample(af.batch_size, af._gen), af.gamma)
    lp = D.td_step(ap.policy_net, ap.target_net, ap.optimizer, ap.replay_buffer.sample(ap.batch_size, ap._gen), ap.gamma)
    assert float(lf) > 0 and torch.equal(lf, lp)


@pytest.mark.gpu
def test_packed_game_at_scale_trains_and_competes(D):
    """16 384 envs with packed replay and a capacity above one decision's transitions: TD steps run (loss > 0), the counters
    agree with the env's, the buffer holds more than one decision's transitions, compete() plays the trained net"""
    from qnet_like import QNetLike
    net = lambda: QNetLike(9, width=16)
    dqn = functools.partial(D.BatchedDQN, replay_size=200_000)
    torch.manual_seed(0)
    B = 16384
    game = D.BatchedGame(D.BatchedEnvCooperation, {"lord": net, "down": None, "up": None}, {"lord": dqn, "down": None, "up": None},
                         train_dict={"lord": True, "down": False, "up": False}, seed=3, num_envs=B, replay="packed")
    rb = game.lord.replay_buffer
    assert isinstance(rb, D.PackedReplayBuffer) and rb.capacity == 200_000
    per_step = 0
    for _ in range(8):
        before = len(rb)
        game.step()
        per_step = max(per_step, len(rb) - before)
    assert per_step > 1000
    hist = game.train(2 * B, log_every=B)
    st = game.env.stats.cpu().numpy()
    assert game.episodes >= 2 * B and game.episodes == st[0] and st[7] == 0
    assert (game.lord_total_wins, game.down_total_wins, game.up_total_wins) == (st[1], st[2], st[3])
    assert any(h["lord"]["mean_loss"] > 0 for h in hist)
    assert len(rb) > per_step
    n = len(rb)
    s0, a0, r, s1, a1, done = rb.decode(torch.arange(n, device="cuda"))
    term = done[:, 0] == 1
    assert term.any() and (~term).any()
    assert (r[:, 0][term].abs() == 100.0).all() and (r[:, 0][~term] == 0).all() and (a1[term] == 0).all()
    wins = D.BatchedGame.compete(D.BatchedEnvCooperation, {"lord": net, "down": None, "up": None},
                                 {"lord": D.BatchedDQN, "down": None, "up": None}, None, total=500, debug=False,
                                 num_envs=256, seed=5, nets={"lord": game.lord.policy_net})
    assert sum(wins.values()) >= 500 and wins["lord"] > 0
