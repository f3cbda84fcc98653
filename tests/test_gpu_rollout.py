"""GPU parity tests of the fused lock-step rollout (ic3net_b200/trainer.py) against
(a) whole episodes recorded from the unmodified reference's Trainer.get_episode
(tests/golden/ep_*.npz) and (b) the oracle replaying every env slot with the same
Philox streams.  Integer outputs (actions, masks, alive) must be identical, rewards
equal float32(reference), float outputs within 1e-5 * max(1,|ref|)."""
import numpy as np
import pytest
import torch

from helpers import finish_args, golden_names, load_golden, make_oracle_env, ns, tj_tables
from oracle import policy as opolicy
from oracle.gen_golden import make_weights
from oracle.rollout import run_episode

pytestmark = pytest.mark.gpu
TOL = 1e-5


def close(a, b, tol=TOL):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.abs(b)))


def cpu(t):
    return t.detach().cpu().numpy()


def build(meta, B, obs_mode="index", use_graph=False, seed=None, env_id0=0, impl=None, **over):
    from ic3net_b200 import data
    from ic3net_b200.comm import CommNetMLP
    from ic3net_b200.trainer import Trainer
    args = ns(meta["args"], nenvs=B, seed=meta["seed"] if seed is None else seed, env_id0=env_id0,
              obs_mode=obs_mode, use_graph=use_graph, policy_impl=impl, **over)
    env = data.init(args.env_name, args)
    finish_args(args, env)
    if impl == "tc" and args.hid_size != 128:
        pytest.skip("tensor-core path is specialised for hid_size 128")
    net = CommNetMLP(args, args.num_inputs)
    sd = make_weights(meta["weights_seed"], args.num_inputs, args.hid_size, args.naction_heads, args.comm_init)
    net.load_state_dict({k: torch.from_numpy(v).float() for k, v in sd.items()})
    return args, env, net, Trainer(args, net, env), opolicy.params_to_f64(sd)


@pytest.mark.parametrize("name", golden_names("ep_"))
@pytest.mark.parametrize("obs_mode", ["index", "dense"])
@pytest.mark.parametrize("impl", ["tc", "simt"])
def test_first_episode_matches_reference_golden(name, obs_mode, impl):
    meta, z = load_golden(name)
    ids = meta["env_ids"]
    B = max(ids) + 1
    args, env, net, tr, p = build(meta, B, obs_mode, impl=impl)
    T = args.max_steps
    batch = tr.rollout(T, meta["epoch"])
    torch.cuda.synchronize()
    for i, env_id in enumerate(ids):
        g = lambda k: z["e%d_%s" % (i, k)]
        L = len(g("act"))
        act = cpu(batch.action)[:L, env_id]
        flips = (act != g("act")) & (g("margin") > 1e-4)
        assert not flips.any(), (name, env_id)
        if not np.array_equal(act, g("act")):
            continue        # an fp32-borderline draw flipped; the teacher-forced test below covers this slot
        assert np.array_equal(cpu(batch.reward)[:L, env_id], g("reward").astype(np.float32))
        assert np.array_equal(cpu(batch.alive_mask)[:L, env_id], g("alive"))
        assert np.array_equal(cpu(batch.episode_mask)[:L, env_id], g("emask")[:, 0])
        assert np.array_equal(cpu(batch.episode_mini_mask)[:L, env_id], g("mini"))
        assert close(cpu(batch.value)[:L, env_id], g("value")), (name, env_id)
        lp = np.concatenate([g("logp%d" % k) for k in range(len(meta["heads"]))], -1)
        assert close(cpu(batch.logp)[:L, env_id], lp), (name, env_id)


@pytest.mark.parametrize("name,B,T", [("ep_pp_easy_ic3net", 11, 70), ("ep_tj_medium_ic3net", 7, 80),
                                      ("ep_tj_easy_ic3net", 9, 45), ("ep_pp_hard_commnet", 3, 90),
                                      ("ep_tj_medium_v1_commnet", 4, 50), ("ep_pp_enemy_ic3net", 9, 50)])
@pytest.mark.parametrize("impl", ["tc", "simt"])
def test_lockstep_rollout_matches_oracle(name, B, T, impl):
    """Every slot, every episode (auto-reset, cut at the batch end), teacher-forced with
    the GPU's own actions so both sides stay on one trajectory; plus the stat sums."""
    meta, z = load_golden(name)
    args, env, net, tr, p = build(meta, B, "index", seed=321, env_id0=50, impl=impl)
    is_tj = args.env_name == "traffic_junction"
    batch = tr.rollout(T, 0)
    stat = tr.collect_stat()
    act, rew = cpu(batch.action), cpu(batch.reward)
    val, lp = cpu(batch.value), cpu(batch.logp)
    emask, mini, alive = cpu(batch.episode_mask), cpu(batch.episode_mini_mask), cpu(batch.alive_mask)
    tot = dict(reward=np.zeros(args.nagents), comm=np.zeros(args.nagents), success=0, episodes=0, flips=0, draws=0)
    for b in range(B):
        t0, k = 0, 0
        orc = make_oracle_env(args, tj_tables(z) if is_tj else None)
        while t0 < T:
            ep = run_episode(orc, p, args, 321, 50 + b, epoch=0, tick0=t0, episode=k,
                             forced_actions=act[t0:, b], max_steps=min(args.max_steps, T - t0))
            L = ep["num_steps"]
            sl = slice(t0, t0 + L)
            assert np.array_equal(rew[sl, b], ep["reward"].astype(np.float32)), (b, k)
            assert np.array_equal(emask[sl, b], ep["emask"][:, 0]) and np.array_equal(mini[sl, b], ep["mini"])
            assert np.array_equal(alive[sl, b], ep["alive"])
            assert close(val[sl, b], ep["value"]) and close(lp[sl, b], ep["logp"]), (b, k)
            # free-running agreement of the sampled actions wherever fp32 cannot flip the draw
            own = np.array([opolicy.sample_actions(np.split(ep["logp"][t], np.cumsum(args.naction_heads)[:-1], -1),
                                                   opolicy.action_draws(321, 50 + b, t0 + t, args.nagents,
                                                                        len(args.naction_heads)))[0]
                            for t in range(L)])
            safe = ep["margin"] > 1e-4
            assert np.array_equal(own[safe], act[sl, b][safe])
            tot["flips"] += int((own != act[sl, b]).sum())
            tot["draws"] += own.size
            tot["reward"] += ep["reward"].sum(0)
            if args.hard_attn:
                tot["comm"] += ep["comm_in"][1:].sum(0) + (act[t0 + L - 1, b, :, -1] if not args.comm_action_one
                                                           else np.ones(args.nagents))
            tot["success"] += max(ep["success"], 0)
            tot["episodes"] += 1
            t0 += L
            k += 1
    assert tot["flips"] <= 1e-3 * tot["draws"]
    assert stat["num_steps"] == B * T and stat["num_episodes"] == tot["episodes"]
    nf = args.nfriendly                   # with --enemy_comm the prey's entries are reported apart (trainer.py:73-75,86-88)
    assert np.allclose(stat["reward"], tot["reward"][:nf], rtol=1e-5, atol=1e-4)
    assert stat["success"] == tot["success"]
    if args.hard_attn:
        assert np.array_equal(stat["comm_action"], tot["comm"][:nf])
    if getattr(args, "enemy_comm", False):
        assert np.allclose(stat["enemy_reward"], tot["reward"][nf:], rtol=1e-5, atol=1e-4)
        assert np.array_equal(stat["enemy_comm"], tot["comm"][nf:])
    else:
        assert "enemy_reward" not in stat and "enemy_comm" not in stat


def test_graph_replay_equals_eager():
    """The graph trainer (warm-up on a rewound snapshot, capture, replay) produces bit for bit what the eager trainer
    produces, rollout after rollout."""
    meta, z = load_golden("ep_tj_medium_ic3net")
    res = {}
    for use_graph in (True, False):
        args, env, net, tr, p = build(meta, 16, "index", use_graph=use_graph, seed=5)
        out = []
        for k in range(3):
            b = tr.rollout(40, 0)
            torch.cuda.synchronize()
            out.append((cpu(b.action).copy(), cpu(b.reward).copy(), cpu(b.value).copy()))
        res[use_graph] = out
    for a, b in zip(res[True], res[False]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])


@pytest.mark.parametrize("name", ["ep_pp_hard_ic3net", "ep_tj_medium_ic3net", "ep_tj_medium_v1_commnet"])
def test_dense_and_index_rollouts_are_identical(name):
    """Dense obs + dense encoder, fused index encoder from the per-position table, fused index encoder without
    the table: bit-identical rollouts (same additions in the same order, include/ic3net_b200.h obs_vocab)."""
    meta, z = load_golden(name)
    if meta["args"]["hid_size"] != 128:
        pytest.skip("fused encoder is part of the tensor-core path (hid_size 128)")
    res = []
    for mode, table in (("index", True), ("index", False), ("dense", True)):
        args, env, net, tr, p = build(meta, 24, mode, seed=77, encoder_table=table)
        b = tr.rollout(30, 0)
        torch.cuda.synchronize()
        assert (tr._xtable is not None) == (mode == "index" and table)
        res.append((cpu(b.action).copy(), cpu(b.value).copy(), cpu(b.reward).copy()))
    for k in (1, 2):
        assert np.array_equal(res[0][0], res[k][0]) and np.array_equal(res[0][1], res[k][1])
        assert np.array_equal(res[0][2], res[k][2])


def test_pp_hard_full_size_rollout_properties():
    """BASELINE c2 at full size (8192 envs): invariants of a 20-step lock-step rollout."""
    meta, z = load_golden("ep_pp_hard_ic3net")
    B, T = 8192, 20
    args, env, net, tr, p = build(meta, B, "index", seed=9)
    b = tr.rollout(T, 0)
    stat = tr.collect_stat()
    assert stat["num_steps"] == B * T
    r = b.reward
    assert bool(((r == 0) | (r == -0.05)).all())                        # mixed mode rewards
    lp = b.logp.double().exp()
    assert torch.allclose(lp[..., :5].sum(-1), torch.ones_like(lp[..., 0]), atol=1e-5)
    assert torch.allclose(lp[..., 5:].sum(-1), torch.ones_like(lp[..., 0]), atol=1e-5)
    assert int(b.action[..., 0].min()) >= 0 and int(b.action[..., 0].max()) <= 4
    assert int(b.action[..., 1].min()) >= 0 and int(b.action[..., 1].max()) <= 1
    assert bool((b.episode_mask[:-1] == 1).all() | (stat["num_episodes"] > B))
    assert bool((b.episode_mask[-1] == 0).all())                         # batch end cuts every open episode
    assert abs(stat["reward"].sum() - float(r.double().sum())) < 1e-2 * B
    assert torch.isfinite(b.value).all()


def replay_slots(args, z, p, batch, slots, T, seed, env_id0):
    """Teacher-forced oracle replay of the given env slots of a lock-step rollout (cut at T)."""
    is_tj = args.env_name == "traffic_junction"
    idx = torch.as_tensor(slots, device=batch.action.device)
    act, rew = cpu(batch.action[:, idx]), cpu(batch.reward[:, idx])
    val, lp = cpu(batch.value[:, idx]), cpu(batch.logp[:, idx])
    emask, mini, alive = cpu(batch.episode_mask[:, idx]), cpu(batch.episode_mini_mask[:, idx]), cpu(batch.alive_mask[:, idx])
    flips = draws = 0
    for j, b in enumerate(slots):
        t0, k = 0, 0
        orc = make_oracle_env(args, tj_tables(z) if is_tj else None)
        while t0 < T:
            ep = run_episode(orc, p, args, seed, env_id0 + b, epoch=0, tick0=t0, episode=k,
                             forced_actions=act[t0:, j], max_steps=min(args.max_steps, T - t0))
            L = ep["num_steps"]
            sl = slice(t0, t0 + L)
            assert np.array_equal(rew[sl, j], ep["reward"].astype(np.float32)), (b, k)
            assert np.array_equal(emask[sl, j], ep["emask"][:, 0]) and np.array_equal(mini[sl, j], ep["mini"]), (b, k)
            assert np.array_equal(alive[sl, j], ep["alive"]), (b, k)
            assert close(val[sl, j], ep["value"]) and close(lp[sl, j], ep["logp"]), (b, k)
            own = np.array([opolicy.sample_actions(np.split(ep["logp"][t], np.cumsum(args.naction_heads)[:-1], -1),
                                                   opolicy.action_draws(seed, env_id0 + b, t0 + t, args.nagents,
                                                                        len(args.naction_heads)))[0]
                            for t in range(L)])
            safe = ep["margin"] > 1e-4
            assert np.array_equal(own[safe], act[sl, j][safe]), (b, k)
            flips += int((own != act[sl, j]).sum())
            draws += own.size
            t0 += L
            k += 1
    assert flips <= 2e-3 * draws


@pytest.mark.parametrize("name,B", [("ep_pp_hard_ic3net", 8192), ("ep_tj_hard_ic3net", 4096)])
def test_full_size_rollout_sampled_slots_match_oracle(name, B):
    """BASELINE c2 / c5 at their FULL batch sizes: 32 env slots drawn at random -- always including the first slot,
    the slots that straddle 128-row tile boundaries of the tensor-core kernels and the very last ones -- are replayed
    step by step through the float64 oracle (bit-exact integers / rewards, 1e-5 on values and log-probs)."""
    meta, z = load_golden(name)
    T, seed, id0 = 24, 4242, 1000
    args, env, net, tr, p = build(meta, B, "index", seed=seed, env_id0=id0)
    batch = tr.rollout(T, 0)
    stat = tr.collect_stat()
    assert stat["num_steps"] == B * T
    N = args.nagents
    rs = np.random.RandomState(7)
    edge = [0, 128 // N, 128 // N + 1, B // 2, B - 2, B - 1, (B * N - 128) // N]       # tile-boundary / tail slots
    slots = sorted(set(edge) | set(int(x) for x in rs.randint(0, B, size=32 - len(set(edge)))))
    replay_slots(args, z, p, batch, slots, T, seed, id0)


@pytest.mark.parametrize("name,impl", [("ep_pp_hard_ic3net", "tc"), ("ep_tj_medium_ic3net", "tc"), ("ep_pp_easy_ic3net", "simt"),
                                       ("ep_tj_medium_v1_commnet", "simt")])
def test_observation_handle_api_is_bit_identical_to_the_dense_tensor_api(name, impl):
    """args.obs_api = 'handle': GymWrapper.reset/step return a LazyObs (ic3net_b200/lazy_obs.py) and CommNetMLP.forward
    evaluates the encoder from the env state; the same public-API loop with dense observation tensors must give the same
    values, log-probs, hidden states and rewards bit for bit, and the handle must materialise the exact dense tensor."""
    from ic3net_b200.action_utils import select_action
    from ic3net_b200.lazy_obs import LazyObs
    meta, z = load_golden(name)
    out = {}
    for api in ("dense", "handle"):
        args, env, net, tr, p = build(meta, 9, "index", seed=77, impl=impl, obs_api=api)
        B, N = 9, args.nagents
        obs = env.reset(0)
        assert isinstance(obs, LazyObs) == (api == "handle")
        hc = net.init_hidden(B)
        info = {"comm_action": torch.zeros(B, N, dtype=torch.uint8, device="cuda")} if args.hard_attn else {}
        rec = []
        for t in range(6):
            if api == "handle" and t == 2:
                dense_now = obs.dense().clone()
            action_out, value, hc = net([obs, hc], info)
            action = select_action(args, action_out)
            obs, reward, done, info_env = env.step([action[..., 0]])
            info = {}
            if args.hard_attn:
                info["comm_action"] = action[..., -1].to(torch.uint8) if not args.comm_action_one else torch.ones(
                    B, N, dtype=torch.uint8, device="cuda")
            if "alive_mask" in info_env:
                info["alive_mask"] = info_env["alive_mask"]
            rec.append((cpu(value).copy(), cpu(torch.cat(action_out, -1)).copy(), cpu(hc[0]).copy(), cpu(reward).copy(),
                        cpu(action).copy()))
            if api == "dense" and t == 1:
                out["dense_obs_t2"] = cpu(obs).copy()
        if api == "handle":
            assert np.array_equal(cpu(dense_now), out["dense_obs_t2"])          # the handle materialises the same tensor
            with pytest.raises(RuntimeError, match="stale"):
                stale = env.reset(0)
                env.step([action[..., 0]])
                stale.dense()
        out[api] = rec
    for a, b in zip(out["dense"], out["handle"]):
        for x, y in zip(a, b):
            assert np.array_equal(x, y)


def test_graph_is_recaptured_when_the_curriculum_moves_the_spawn_rate():
    """Kernel arguments passed by value (ic3_tj_cfg.spawn_thr) are frozen into a captured CUDA graph; the traffic-junction
    curriculum (traffic_junction_env.py:196-200,620-626) changes that value between epochs.  The graph trainer must follow:
    its rollouts equal an eager trainer's, epoch after epoch, and its add_rate statistic is the one the kernels used."""
    meta, z = load_golden("ep_tj_medium_ic3net")
    over = dict(add_rate_min=0.05, add_rate_max=0.5, curr_start=0, curr_end=4)
    res = {}
    for use_graph in (False, True):
        args, env, net, tr, p = build(meta, 16, "index", use_graph=use_graph, seed=5, **over)
        out = []
        for epoch in (0, 1, 2, 3, 3, 6):
            b = tr.rollout(20, epoch)
            st = tr.collect_stat()
            out.append((cpu(b.action).copy(), cpu(b.reward).copy(), cpu(b.alive_mask).copy(), st["add_rate"] / max(1, st["num_episodes"]),
                        int(env.env.cfg.spawn_thr)))
        res[use_graph] = out
    rates = [o[3] for o in res[True]]
    assert rates[0] < rates[1] < rates[2] < rates[3] == rates[4]            # the schedule really moved
    for a, b in zip(res[False], res[True]):
        assert a[3] == b[3] and a[4] == b[4]
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2])
    alive_first, alive_last = res[True][0][2].mean(), res[True][3][2].mean()
    assert alive_last > alive_first                                          # more cars at the higher add_rate
