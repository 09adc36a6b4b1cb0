"""Batched rollout / trainer driver with the reference's `Game` and `DQNFirst` surface (SURVEY.md 8f rank 2).

Reference: game.py:10-275 (`Game`: step / feedback / lord_turn / down_turn / up_turn / play / train / compete) drives ONE
env through one decision at a time; dqn.py:10-80 (`DQNFirst`) owns policy / target net, the optimizer, epsilon and a
`deque` replay buffer, and `perceive` appends one transition and does one TD step.  Here one `step()` is one decision of
EVERY env of a `BatchedEnv*`: roles that have an agent score all their legal moves in one batched forward and pick
(epsilon-)greedily (`BatchedGreedyPolicy` + ddz_select_actions), the transitions of the learning roles are assembled on
the device with the reference's delayed-feedback rule (`TransitionCollector`), and `BatchedDQN.perceive` appends the
whole batch to a GPU ring buffer and does the reference's TD step.

Differences, all forced by the scope (DESIGN.md 1): a role WITHOUT a network plays uniformly random legal moves
(`step_random`, envi.py:79-85) -- the reference's rule bot behind `step_auto` is the absent native RHCP code; an
"episode" is one finished game of any env, so `train(episodes)` runs until that many games have ended; shuffles are
host-made deals handed to `prepare` (a pool that finished envs re-deal from).
"""
import collections
import math
import time

import torch

from .agent import BatchedGreedyPolicy
from .env import VARIANT_CHANNELS, random_deals
from .policy import HeadedPolicy, _sample as policy_sample
from .trainer import PackedReplayBuffer, ReplayBuffer, TransitionCollector, td_step

# config.py:7-14
GAMMA = 0.95
EPSILON_HIGH = 0.5
EPSILON_LOW = 0.01
REPLAY_SIZE = 20000
BATCH_SIZE = 256
DECAY = int((8000 * (2 / 3)) / 5)
UPDATE_TARGET_EVERY = 20

ROLES = ("up", "lord", "down")            # seat index 0 / 1 / 2 (envi.py:23-24)
ROLE_INDEX = {r: i for i, r in enumerate(ROLES)}


class BatchedDQN:
    """dqn.py:10-80 over batches: same attributes (`epsilon`, `replay_buffer`, `policy_net`, `target_net`, `optimizer`)
    and verbs (`perceive`, `e_greedy_action`, `greedy_action`, `update_epsilon`, `update_target`)."""

    def __init__(self, net_cls, face_channels, device, replay_size=REPLAY_SIZE, batch_size=BATCH_SIZE, gamma=GAMMA,
                 lr=1e-4, decay=DECAY, update_target_every=UPDATE_TARGET_EVERY, seed=0, fused=False, precision="fp32",
                 replay="float"):
        """fused=True: the moves are scored by agent.FusedQScorer (ddz_q_features + two GEMMs, for the NetComplicated family of
        net.py) instead of the module's forward; its tables are rebuilt from the weights after every update.
        replay="packed": the replay buffer is a trainer.PackedReplayBuffer (transitions as packed states and moves, 176 B
        each; perceive takes what TransitionCollector(packed=True) emits); "float" (default): trainer.ReplayBuffer."""
        self.device = torch.device(device)
        self.epsilon = EPSILON_HIGH
        self.batch_size, self.gamma, self.decay, self.update_target_every = int(batch_size), float(gamma), decay, update_target_every
        self.policy_net = net_cls().to(self.device)
        self.target_net = net_cls().to(self.device)
        self.target_net.load_state_dict(self.policy_net.state_dict())
        self.optimizer = torch.optim.Adam(self.policy_net.parameters(), lr)
        if replay == "packed":
            self.replay_buffer = PackedReplayBuffer(replay_size, VARIANT_CHANNELS.index(face_channels), self.device)
        elif replay == "float":
            self.replay_buffer = ReplayBuffer(replay_size, face_channels, self.device)
        else:
            raise ValueError("replay must be 'float' or 'packed', not %r" % (replay,))
        self._policy = BatchedGreedyPolicy(self.policy_net, epsilon=0.0, seed=seed, fused=fused, precision=precision)
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed(int(seed) + 1)

    def q_values(self, env, env_mask=None):
        return self._policy.q_values(env, env_mask)

    def e_greedy_action(self, env, q):
        """int32 [B] list index per env: argmax Q, or a uniform random legal move with probability epsilon (dqn.py:50-61)"""
        self._policy.epsilon = self.epsilon
        return self._policy.select(env, q)

    def greedy_action(self, env, q):
        """int32 [B] list index per env: argmax Q (dqn.py:63-71)"""
        self._policy.epsilon = 0.0
        return self._policy.select(env, q)

    def perceive(self, s0, a0, r, s1, a1, done, updates=1):
        """append a batch of transitions; once the buffer holds a minibatch, `updates` TD steps (dqn.py:21-48).
        Returns the last loss as a float tensor on the device, or None."""
        self.replay_buffer.append(s0, a0, r, s1, a1, done)
        if len(self.replay_buffer) < self.batch_size or s0.shape[0] == 0:
            return None
        loss = None
        for _ in range(updates):
            loss = td_step(self.policy_net, self.target_net, self.optimizer,
                           self.replay_buffer.sample(self.batch_size, self._gen), self.gamma)
        if self._policy.scorer is not None:
            self._policy.scorer.refresh()                      # the weights moved: rebuild the scoring tables
        return loss

    def update_epsilon(self, episode):
        self.epsilon = EPSILON_LOW + (EPSILON_HIGH - EPSILON_LOW) * math.exp(-1.0 * episode / self.decay)   # dqn.py:73-76

    def update_target(self, episode):
        if episode % self.update_target_every == 0:                                                     # dqn.py:78-80
            self.target_net.load_state_dict(self.policy_net.state_dict())


class BatchedGame:
    """game.py:10-238 over a batched env.  nets_dict / dqns_dict / reward_dict / train_dict / preload keep the
    reference's meaning (role -> net class / DQN class / terminal reward magnitude / keep training / checkpoint path);
    `dqns_dict[role]` is called as `dqn_cls(net_cls, face_channels, device)` (BatchedDQN's signature).
    search_dict (optional) seats the search bot: role -> keyword arguments of search.pimc_search, e.g.
    {"lord": {"determinizations": 8, "computation_budget": 125}}; that role plays from its own view (determinized UCT),
    or with "determinizations": 0 the full-information search.uct_search, which sees every hand.
    policy_dict (optional) seats a fixed-head policy: role -> a module (on the game's device) that maps the env's face
    [B, C, 15, 4] to logits [B, 13551] over the action ids; that role samples its move from the softmax over its legal ids
    (policy.policy_sample) at temperature `policy_temperature` (1.0; compete plays 0, the argmax).  A policy.HeadedPolicy
    (trunk + LinearPolicyHead) is sampled through head.sample(env, trunk(face)), without the dense logits.  Learning stays
    with the caller.  A role has a net, a search entry or a policy entry, never two.
    replay="packed" keeps the learning roles' transitions as packed states and moves (trainer.PackedReplayBuffer, 176 B a
    transition instead of 2 * 240 * (C + 1) + 8 B): `dqns_dict[role]` is then called with the extra keyword replay="packed".
    Set the capacity through the DQN class, e.g. functools.partial(BatchedDQN, replay_size=10_000_000)."""

    def __init__(self, env_cls, nets_dict, dqns_dict, reward_dict=None, train_dict=None, preload=None, seed=None,
                 debug=False, num_envs=4096, pool_games=8, deals=None, device=None, updates_per_step=1, search_dict=None,
                 replay="float", policy_dict=None):
        if reward_dict is None:
            reward_dict = {"lord": 100, "down": 50, "up": 50}
        if train_dict is None:
            train_dict = {"lord": True, "down": True, "up": True}
        preload = preload or {}
        assert not (nets_dict.keys() ^ dqns_dict.keys()), "Net and DQN must match"
        if replay not in ("float", "packed"):
            raise ValueError("replay must be 'float' or 'packed', not %r" % (replay,))
        self.packed = replay == "packed"
        self.search_dict = {r: dict(kw) for r, kw in (search_dict or {}).items()}
        for role in self.search_dict:
            if role not in ROLE_INDEX:
                raise ValueError("unknown role %r in search_dict" % (role,))
            if nets_dict.get(role):
                raise ValueError("role %r has both a net and a search entry" % (role,))
        self.policy_dict = dict(policy_dict or {})
        for role in self.policy_dict:
            if role not in ROLE_INDEX:
                raise ValueError("unknown role %r in policy_dict" % (role,))
            if nets_dict.get(role) or role in self.search_dict:
                raise ValueError("role %r has a policy entry and a net or search entry" % (role,))
        self.policy_temperature = 1.0
        self._search_seed = int(seed) if seed else 0
        self.env = env_cls(num_envs, debug=debug, seed=seed, device=device)
        self.B, self.device = self.env.B, self.env.device
        self.reward_dict, self.train_dict, self.preload = reward_dict, train_dict, preload
        self.updates_per_step = int(updates_per_step)
        self.lord = self.down = self.up = None
        self.lord_train = self.down_train = self.up_train = False
        self._collectors = {}
        for role in ("lord", "down", "up"):
            if nets_dict.get(role):
                extra = {"replay": "packed"} if self.packed else {}      # custom DQN classes keep their signature
                agent = dqns_dict[role](nets_dict[role], self.env.C, self.device, **extra)
                setattr(self, role, agent)
                setattr(self, "%s_train" % role, bool(train_dict.get(role)))
                if preload.get(role):
                    for net in (agent.target_net, agent.policy_net):
                        net.load(preload[role])
                if train_dict.get(role):
                    self._collectors[role] = TransitionCollector(self.env, role=ROLE_INDEX[role],
                                                                 reward=float(reward_dict[role]),
                                                                 **({"packed": True} if self.packed else {}))
        # counters with the reference's names (game.py:20-26)
        self.lord_wins, self.down_wins, self.up_wins = [], [], []
        self.up_total_wins = self.lord_total_wins = self.down_total_wins = 0
        self.up_recent_wins = self.lord_recent_wins = self.down_recent_wins = 0
        self.lord_total_loss = self.down_total_loss = self.up_total_loss = 0.0
        self.lord_loss_count = self.down_loss_count = self.up_loss_count = 0
        self.episodes = 0
        self.iterations = 0
        self._gen = torch.Generator(device=self.device)
        self._gen.manual_seed((int(seed) if seed else 0) + 12345)
        self.pool_games = int(pool_games)
        self._deal_seed = (int(seed) if seed else 0) + 777
        self._own_deals = deals is None                  # caller-supplied deals are a closed set by the caller's choice
        if deals is None:
            deals = random_deals(self.B, seed=self._deal_seed, pool_games=self.pool_games)
        self._perm = torch.as_tensor(deals[0]).to(self.device).reshape(self.pool_games, self.B, 54).contiguous()
        self._lord_pile = torch.as_tensor(deals[1]).to(self.device).reshape(self.pool_games, self.B).contiguous()
        self._slots_made = self.pool_games               # deal number j of every env lives in slot j % pool_games
        self.env.prepare(self._perm, self._lord_pile, pool_games=self.pool_games)

    def _refresh_pool(self):
        """The reference shuffles a fresh deck for every game (game.py:170-171).  Env b takes row (deals consumed % pool) of
        the device-resident pool, so a slot every env has passed is replaced by new host-made deals (seeded by its deal
        number): no env ever replays a deal, however long the run."""
        if not self._own_deals:
            return
        passed = int((self.env._fields()[1] >> 8).min().item())      # deals consumed by the slowest env
        while self._slots_made - self.pool_games < passed - 1:       # slot of deal number j - pool is no longer needed
            j = self._slots_made
            perm, lord = random_deals(self.B, seed=self._deal_seed + 7919 * j)
            self._perm[j % self.pool_games].copy_(torch.as_tensor(perm), non_blocking=False)
            self._lord_pile[j % self.pool_games].copy_(torch.as_tensor(lord), non_blocking=False)
            self._slots_made += 1

    # ------------------------------------------------------------------ one decision of every env
    def accumulate_loss(self, name, loss):
        assert name in {"up", "down", "lord"}
        if loss is not None:
            setattr(self, "%s_loss_count" % name, getattr(self, "%s_loss_count" % name) + 1)
            setattr(self, "%s_total_loss" % name, getattr(self, "%s_total_loss" % name) + float(loss))

    def reset_recent(self):
        self.lord_recent_wins = self.up_recent_wins = self.down_recent_wins = 0
        self.lord_total_loss = self.down_total_loss = self.up_total_loss = 0.0
        self.lord_loss_count = self.down_loss_count = self.up_loss_count = 0

    def step(self):
        """Game.step + Game.feedback for the seat to move in every env (game.py:90-127), then re-deal of finished envs
        (Game.play's reset/prepare, game.py:170-171).  Returns the number of games that ended with this decision."""
        env, B, dev = self.env, self.B, self.device
        acts, offs = env.valid_actions()
        off = offs.to(torch.int64)
        cnt = off[1:] - off[:-1]
        seat = env.get_role_ID() - 1
        live = ~env.is_done
        choice = torch.randint(0, 1 << 30, (B,), device=dev, generator=self._gen) % cnt.clamp(min=1)   # step_random
        last = max(int(acts.shape[0]) - 1, 0)
        pending = []
        for role in ("lord", "down", "up"):
            agent = getattr(self, role)
            if agent is None:
                continue
            mine = (seat == ROLE_INDEX[role]) & live
            q = agent.q_values(env, mine)
            training = getattr(self, "%s_train" % role)
            k = (agent.e_greedy_action(env, q) if training else agent.greedy_action(env, q)).to(torch.int64)
            choice = torch.where(mine, k.clamp(min=0), choice)
            if training:
                kg = agent.greedy_action(env, q).to(torch.int64).clamp(min=0)
                if self.packed:                      # packed moves, 0 (a pass row of zeros) where there is no move
                    au, keep = env.actions_packed, cnt > 0
                    a0 = au[(off[:-1] + k.clamp(min=0)).clamp(max=last)] * keep
                    a1 = au[(off[:-1] + kg).clamp(max=last)] * keep
                else:
                    keep = (cnt > 0)[:, None, None]
                    a0 = acts[(off[:-1] + k.clamp(min=0)).clamp(max=last)] * keep
                    a1 = acts[(off[:-1] + kg).clamp(max=last)] * keep
                pending.append((role, self._collectors[role].on_turn(a0, a1)))
        for role, kw in self.search_dict.items():
            mine = (seat == ROLE_INDEX[role]) & live
            if bool(mine.any()):
                choice = torch.where(mine, self._search(kw, mine).to(torch.int64).clamp(min=0), choice)
        for role, module in self.policy_dict.items():
            mine = (seat == ROLE_INDEX[role]) & live
            if bool(mine.any()):
                # record=False: a -1 (nothing to draw from) is counted once, as the step's illegal choice
                if isinstance(module, HeadedPolicy):              # the head at the legal ids only, no dense logits
                    with torch.no_grad():
                        h = module.trunk(env.face)
                    k = module.head._sample(env, h, self.policy_temperature, self._search_seed, mine, record=False)[0]
                else:
                    with torch.no_grad():
                        logits = module(env.face)
                    k = policy_sample(env, logits, self.policy_temperature, self._search_seed, mine, record=False)[0]
                choice = torch.where(mine, k.to(torch.int64), choice)
        was_done = env.is_done.clone()
        env.step(choice.to(torch.int32))
        env.observe()
        newly = env.is_done & ~was_done
        for role, tr in pending:
            self.accumulate_loss(role, getattr(self, role).perceive(*tr[:6], updates=self.updates_per_step))
        for role, col in self._collectors.items():
            self.accumulate_loss(role, getattr(self, role).perceive(*col.on_step_done(newly)[:6],
                                                                    updates=self.updates_per_step))
        winner = env.winner[newly]
        ended = int(newly.sum().item())
        if ended:
            w = torch.bincount(winner.to(torch.int64), minlength=3).tolist()
            for role in ROLES:
                n = w[ROLE_INDEX[role]]
                setattr(self, "%s_total_wins" % role, getattr(self, "%s_total_wins" % role) + n)
                setattr(self, "%s_recent_wins" % role, getattr(self, "%s_recent_wins" % role) + n)
            if self.iterations % 16 == 0:
                self._refresh_pool()
            env.prepare(self._perm, self._lord_pile, only_done=True, pool_games=self.pool_games)
        self.episodes += ended
        self.iterations += 1
        return ended

    def _search(self, kw, mine):
        """the search seat's choice for the envs of `mine`: pimc_search, or uct_search for determinizations = 0; the seed is
        derived from (seed, iterations), so every decision draws afresh and a run is reproducible"""
        from .search import pimc_search, uct_search
        kw = dict(kw)
        D = int(kw.pop("determinizations", 16))
        seed = (self._search_seed * 1000003 + self.iterations + 1) & (2 ** 64 - 1)
        if D == 0:
            return uct_search(self.env, seed=seed, env_mask=mine, **kw)[0]
        return pimc_search(self.env, determinizations=D, seed=seed, env_mask=mine, **kw)[0]

    def play(self, games=None):
        """decisions until `games` more games have ended (default: one per env, the batched `Game.play`)"""
        target = self.episodes + (self.B if games is None else int(games))
        while self.episodes < target:
            self.step()

    # ------------------------------------------------------------------ training loop (game.py:183-238)
    def train(self, episodes, log_every=100, model_every=1000, logger=None):
        if not any(getattr(self, r) and getattr(self, "%s_train" % r) for r in ROLES):
            print("No agent need train.")
            return []
        history, start, next_log, next_model, recent0 = [], time.time(), log_every, model_every, 0
        end = self.episodes + int(episodes)
        while self.episodes < end:
            self.step()
            for role in ROLES:
                ai = getattr(self, role)
                if ai:                      # the schedules tick once per decision of the whole batch
                    ai.update_epsilon(self.iterations)
                    ai.update_target(self.iterations)
            if self.episodes >= next_log:
                n = max(1, self.episodes - recent0)
                rec = {"episodes": self.episodes, "iterations": self.iterations, "seconds": time.time() - start}
                for role in ROLES:
                    rec[role] = {"recent_win": getattr(self, "%s_recent_wins" % role) / n,
                                 "total_win": getattr(self, "%s_total_wins" % role) / max(1, self.episodes),
                                 "mean_loss": getattr(self, "%s_total_loss" % role) /
                                              (getattr(self, "%s_loss_count" % role) + 1e-3)}
                history.append(rec)
                if logger:
                    logger.info(str(rec))
                self.lord_wins.append(self.lord_recent_wins); self.up_wins.append(self.up_recent_wins)
                self.down_wins.append(self.down_recent_wins)
                self.reset_recent()
                recent0, start = self.episodes, time.time()
                while next_log <= self.episodes:
                    next_log += log_every
            if self.episodes >= next_model:
                for role in ROLES:
                    ai = getattr(self, role)
                    if ai and hasattr(ai.policy_net, "save"):
                        ai.policy_net.save("%s_%d" % (role, self.episodes))
                while next_model <= self.episodes:
                    next_model += model_every
        return history

    # ------------------------------------------------------------------ evaluation (game.py:240-275)
    @staticmethod
    def compete(env_cls, nets_dict, dqns_dict, model_dict, total=1000, print_every=100, debug=True, num_envs=4096,
                seed=None, device=None, nets=None, search_dict=None, policy_dict=None):
        """greedy play of the given networks (others random) until `total` games have ended; Counter of wins per role.
        `nets` may hand over already constructed networks per role instead of checkpoints in model_dict; search_dict
        seats the search bot and policy_dict a fixed-head policy as in BatchedGame (played at temperature 0: argmax)."""
        assert not (nets_dict.keys() ^ dqns_dict.keys()), "Net and DQN must match"
        train_dict = {r: False for r in ROLES}
        game = BatchedGame(env_cls, nets_dict, dqns_dict, train_dict=train_dict, preload=model_dict or {}, seed=seed,
                           debug=False, num_envs=num_envs, device=device, search_dict=search_dict, policy_dict=policy_dict)
        game.policy_temperature = 0.0
        for role, net in (nets or {}).items():
            getattr(game, role).policy_net.load_state_dict(net.state_dict())
        wins = collections.Counter()
        next_print = print_every
        while game.episodes < total:
            game.step()
            if debug and game.episodes >= next_print:
                print("Reach at %d: up %.2f%% lord %.2f%% down %.2f%%" % (
                    game.episodes, 100 * game.up_total_wins / game.episodes, 100 * game.lord_total_wins / game.episodes,
                    100 * game.down_total_wins / game.episodes))
                while next_print <= game.episodes:
                    next_print += print_every
        for role in ROLES:
            wins[role] = getattr(game, "%s_total_wins" % role)
        return wins
