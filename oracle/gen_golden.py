"""Generate tests/golden/*.npz by running the UNMODIFIED reference in this container.

TEST INFRASTRUCTURE.  Run:  python -m oracle.gen_golden   (needs /root/reference)

For every case the reference (float64, B=1) is driven through its own public
surface -- ``GymWrapper.reset/step``, ``CommNetMLP.forward``, and the literal
``Trainer.get_episode`` loop (trainer.py:26-126) -- with its random draws routed
to the shared Philox streams (oracle/philox.py):
  * PP spawn   np.random.choice(D*D, N+1, replace=False)  predator_prey_env.py:174
  * TJ spawn   np.random.uniform / np.random.choice       traffic_junction_env.py:375,383,618
  * actions    torch.multinomial                          action_utils.py:35
Before anything is written the oracle restatement is asserted to reproduce the
reference bit-for-bit (integers, masks, observations) / to 1e-12 (float64 policy
outputs).  The fixtures are then what tests compare oracle and CUDA against on
machines that have no /root/reference.
"""
import json
import os
import sys

import numpy as np

from . import philox, policy, pp_env, ref_shims, tj_env

GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


# --------------------------------------------------------------------------
# deterministic weights (numpy legacy MT19937 is stable across versions)
# --------------------------------------------------------------------------
def make_weights(seed, obs_dim, hid, heads, comm_init="uniform"):
    """state_dict-shaped float64 arrays, U(-1/sqrt(fan_in), 1/sqrt(fan_in)) like
    torch's default nn.Linear / nn.LSTMCell init (values differ, law is the same)."""
    rs = np.random.RandomState(seed)

    def U(shape, fan_in):
        b = 1.0 / np.sqrt(fan_in)
        return rs.uniform(-b, b, size=shape)

    sd = {}
    for k, na in enumerate(heads):
        sd["heads.%d.weight" % k] = U((na, hid), hid)
        sd["heads.%d.bias" % k] = U((na,), hid)
    sd["encoder.weight"] = U((hid, obs_dim), obs_dim)
    sd["encoder.bias"] = U((hid,), obs_dim)
    sd["hidd_encoder.weight"] = U((hid, hid), hid)
    sd["hidd_encoder.bias"] = U((hid,), hid)
    sd["f_module.weight_ih"] = U((4 * hid, hid), hid)
    sd["f_module.weight_hh"] = U((4 * hid, hid), hid)
    sd["f_module.bias_ih"] = U((4 * hid,), hid)
    sd["f_module.bias_hh"] = U((4 * hid,), hid)
    sd["C_modules.0.weight"] = U((hid, hid), hid) if comm_init != "zeros" else np.zeros((hid, hid))
    sd["C_modules.0.bias"] = U((hid,), hid)
    sd["value_head.weight"] = U((1, hid), hid)
    sd["value_head.bias"] = U((1,), hid)
    return sd


# --------------------------------------------------------------------------
# reference-side RNG routing
# --------------------------------------------------------------------------
class RefRandom(object):
    """Routes the reference's draws to Philox(seed, env_id, tick, stream, index)."""

    def __init__(self, seed, env_id):
        self.seed, self.env_id = seed, env_id
        self.tick = 0          # env step counter (TJ spawn + action streams)
        self.episode = 0       # PP reset stream
        self.group = -1        # arrival group of the last np.random.uniform() call
        self.sub = 0
        self.head = 0
        self.margins = []

    # numpy side ---------------------------------------------------------------
    def uniform(self, *a, **k):
        assert not a and not k
        self.group += 1
        self.sub = 1
        self._w = philox.draw_u24(self.seed, self.env_id, self.tick, philox.STREAM_TJ_SPAWN, self.group)
        return float(self._w[0]) * 2.0 ** -24

    def choice(self, a, size=None, replace=True, p=None):
        if replace is False:                       # PP spawn (predator_prey_env.py:174)
            ncell, need = int(a), int(size)
            cells, blk = [], 0
            while len(cells) < need:
                for w in philox.draw_u24(self.seed, self.env_id, self.episode, philox.STREAM_PP_RESET, blk):
                    cell = int((int(w) * ncell) >> 24)
                    if cell not in cells:
                        cells.append(cell)
                        if len(cells) == need:
                            break
                blk += 1
            return np.array(cells)
        arr = np.arange(a) if np.isscalar(a) else np.asarray(a)
        w = int(self._w[self.sub])
        self.sub += 1
        return arr[(w * len(arr)) >> 24]

    # torch side ---------------------------------------------------------------
    def multinomial(self, probs, num_samples):
        import torch
        assert num_samples == 1
        pr = probs.detach().numpy()
        out = np.zeros((pr.shape[0], 1), dtype=np.int64)
        for i in range(pr.shape[0]):
            u24 = int(philox.draw_u24(self.seed, self.env_id, self.tick, philox.STREAM_ACTION, i)[self.head])
            u = u24 * 2.0 ** -24
            cdf = np.cumsum(pr[i])
            a = len(cdf) - 1
            for k in range(len(cdf)):
                if cdf[k] > u:
                    a = k
                    break
            out[i, 0] = a
        self.head += 1
        return torch.from_numpy(out)


class routed(object):
    def __init__(self, rr):
        self.rr = rr

    def __enter__(self):
        import torch
        self._s = (np.random.uniform, np.random.choice, torch.multinomial)
        np.random.uniform, np.random.choice, torch.multinomial = self.rr.uniform, self.rr.choice, self.rr.multinomial
        return self.rr

    def __exit__(self, *e):
        import torch
        np.random.uniform, np.random.choice, torch.multinomial = self._s
        return False


# --------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------
def tj_tables_from_ref(env):
    routes = [[np.asarray(p, dtype=np.int64) for p in grp] for grp in env.routes]
    return {"grid": np.asarray(env.grid, dtype=np.int64), "routes": routes}


def pack_routes(routes):
    """-> (route_len [G,P], route_cells [G,P,Lmax,2]) padded with -1."""
    G, P = len(routes), len(routes[0])
    L = max(len(p) for g in routes for p in g)
    ln = np.zeros((G, P), dtype=np.int64)
    cells = -np.ones((G, P, L, 2), dtype=np.int64)
    for g, grp in enumerate(routes):
        assert len(grp) == P
        for k, p in enumerate(grp):
            ln[g, k] = len(p)
            cells[g, k, :len(p)] = p
    return ln, cells


def unpack_routes(ln, cells):
    return [[cells[g, k, :ln[g, k]] for k in range(ln.shape[1])] for g in range(ln.shape[0])]


def save(name, meta, **arrays):
    os.makedirs(GOLDEN, exist_ok=True)
    path = os.path.join(GOLDEN, name + ".npz")
    np.savez_compressed(path, meta=np.array(json.dumps(meta)), **arrays)
    print("wrote %-40s %7.1f KB" % (name + ".npz", os.path.getsize(path) / 1024.0))


def make_oracle_env(args, tables=None):
    if args.env_name == "predator_prey":
        return pp_env.PredatorPreyOracle(args.nfriendly, args.dim, args.vision, args.mode,
                                         args.nenemies, args.no_stay, getattr(args, "enemy_comm", False))
    return tj_env.TrafficJunctionOracle(args.nagents, args.dim, args.vision, args.difficulty, tables,
                                        args.add_rate_min, args.add_rate_max, args.curr_start, args.curr_end)


# --------------------------------------------------------------------------
# 1. TJ static tables
# --------------------------------------------------------------------------
def gen_tj_tables():
    cases = [("easy", d) for d in (6, 8, 10)] + [("medium", d) for d in (6, 8, 10, 14, 16)] + \
            [("hard", d) for d in (9, 12, 15, 18, 21)]
    for diff, dim in cases:
        for vision in (0,):
            a = ref_shims.make_args(env_name="traffic_junction", nagents=4, dim=dim, vision=vision,
                                    difficulty=diff, ic3net=True)
            try:
                env = ref_shims.make_ref_env(a).env
            except Exception as e:  # reference walker can fail on tiny boards
                print("reference cannot build tj %s dim=%d: %r" % (diff, dim, e))
                continue
            t = tj_tables_from_ref(env)
            ln, cells = pack_routes(t["routes"])
            dims, base, outside, car, vocab, npath = tj_env.constants(diff, dim)
            assert tuple(env.dims) == tuple(dims) and env.BASE == base and env.OUTSIDE_CLASS == outside
            assert env.CAR_CLASS == car and env.vocab_size == vocab and env.npath == npath
            save("tj_tables_%s_%d" % (diff, dim),
                 dict(difficulty=diff, dim=dim, dims=list(map(int, dims)), BASE=base, OUTSIDE=outside, CAR=car,
                      vocab=vocab, npath=npath),
                 grid=t["grid"], route_len=ln, route_cells=cells)


# --------------------------------------------------------------------------
# 2. env-only trajectories (random actions)
# --------------------------------------------------------------------------
def gen_env_case(name, T, seed, env_id, store_obs=True, **kw):
    args = ref_shims.make_args(**kw)
    w = ref_shims.make_ref_env(args)
    env = w.env
    tables = tj_tables_from_ref(env) if args.env_name == "traffic_junction" else None
    orc = make_oracle_env(args, tables)
    is_tj = args.env_name == "traffic_junction"
    rr = RefRandom(seed, env_id)
    ars = np.random.RandomState(seed + 77)
    rec = dict(obs=[], reward=[], done=[], act=[], loc=[], aux=[], alive=[], completed=[])
    with routed(rr):
        obs = w.reset(0)
    if is_tj:
        oobs = orc.reset(0)
    else:
        oobs = orc.flat_obs(orc.reset(seed=seed, env_id=env_id, episode=0))
        assert np.array_equal(orc.predator_loc, env.predator_loc) and np.array_equal(orc.prey_loc, env.prey_loc)
    assert np.array_equal(obs.numpy()[0], oobs), name + ": reset obs"
    rec["obs0"] = obs.numpy()[0].copy()
    rec["loc0"] = (np.array(env.car_loc) if is_tj else np.vstack([env.predator_loc, env.prey_loc])).copy()
    for t in range(T):
        act = ars.randint(0, env.naction, size=args.nagents)
        rr.group, rr.head = -1, 0
        with routed(rr):
            obs, r, done, info = w.step([act])
        if is_tj:
            oo, orr, od, oi = orc.step(act, seed=seed, env_id=env_id)
            assert orc.tick == rr.tick + 1
            loc = np.array(env.car_loc)
            assert np.array_equal(loc, orc.car_loc), name
            assert np.array_equal(info["alive_mask"], oi["alive_mask"])
            assert np.array_equal(info["is_completed"], oi["is_completed"])
            assert np.array_equal(np.asarray(env.wait), orc.wait)
            assert np.array_equal(np.asarray(env.route_id), orc.route_id)
            assert np.array_equal(np.asarray(env.car_last_act), orc.last_act)
            assert env.has_failed == orc.has_failed and env.cars_in_sys == orc.cars_in_sys
            aux = np.stack([np.asarray(env.wait, dtype=np.int64), np.asarray(env.route_id, dtype=np.int64),
                            np.asarray(env.car_last_act, dtype=np.int64),
                            np.asarray(env.car_route_loc, dtype=np.int64)], 1)
            rec["alive"].append(info["alive_mask"].copy())
            rec["completed"].append(info["is_completed"].copy())
        else:
            oo, orr, od, oi = orc.step(act)
            oo = orc.flat_obs(oo)
            loc = np.vstack([env.predator_loc, env.prey_loc])
            assert np.array_equal(env.predator_loc, orc.predator_loc), name
            assert np.array_equal(env.reached_prey, orc.reached)
            assert env.stat.get("success") == orc.stat.get("success")
            aux = np.asarray(env.reached_prey, dtype=np.int64)[:, None]
            rec["alive"].append(np.ones(args.nagents))
            rec["completed"].append(np.zeros(args.nagents))
        rr.tick += 1
        assert np.array_equal(obs.numpy()[0], oo), "%s: obs t=%d" % (name, t)
        assert np.array_equal(r, orr), "%s: reward t=%d" % (name, t)
        assert done == od
        rec["obs"].append(obs.numpy()[0].copy())
        rec["reward"].append(np.asarray(r, dtype=np.float64).copy())
        rec["done"].append(int(done))
        rec["act"].append(act.copy())
        rec["loc"].append(loc.copy())
        rec["aux"].append(aux.copy())
        if done:
            break
    meta = dict(kind="env", seed=seed, env_id=env_id, args={k: v for k, v in vars(args).items()
                                                            if isinstance(v, (int, float, str, bool))},
                obs_dim=int(w.observation_dim), success=int(env.stat.get("success", -1)))
    arrays = dict(obs0=rec["obs0"], loc0=rec["loc0"], reward=np.array(rec["reward"]), done=np.array(rec["done"]),
                  act=np.array(rec["act"]), loc=np.array(rec["loc"]), aux=np.array(rec["aux"]),
                  alive=np.array(rec["alive"]), completed=np.array(rec["completed"]))
    if store_obs:
        arrays["obs"] = np.array(rec["obs"]).astype(np.float32)
    if is_tj:
        arrays["grid"] = tables["grid"]
        arrays["route_len"], arrays["route_cells"] = pack_routes(tables["routes"])
    save(name, meta, **arrays)


# --------------------------------------------------------------------------
# 3. policy forward (single step, random inputs)
# --------------------------------------------------------------------------
def gen_forward_case(name, seed, obs_dim, heads, use_alive, nrep=4, **kw):
    import torch
    torch.set_default_dtype(torch.float64)
    ref_shims.install()
    from comm import CommNetMLP
    args = ref_shims.make_args(**kw)
    args.naction_heads, args.continuous = list(heads), False
    args.num_actions, args.dim_actions = list(heads), len(heads)
    args.recurrent, args.rnn_type = True, "LSTM"
    net = CommNetMLP(args, obs_dim)
    sd = make_weights(seed, obs_dim, args.hid_size, heads, args.comm_init)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    rs = np.random.RandomState(seed + 1)
    n, H = args.nagents, args.hid_size
    out = dict(obs=[], h=[], c=[], comm=[], alive=[], value=[], h2=[], c2=[], x=[])
    for k in range(len(heads)):
        out["logp%d" % k] = []
    for rep in range(nrep):
        obs = np.zeros((n, obs_dim))
        nz = rs.randint(0, obs_dim, size=(n, min(8, obs_dim)))
        for i in range(n):
            obs[i, nz[i]] = rs.randint(1, 4, size=nz.shape[1])
        if rep == nrep - 1:
            obs = rs.uniform(-1, 1, size=(n, obs_dim))          # a fully dense observation
        h = rs.uniform(-1, 1, size=(n, H)) if rep else np.zeros((n, H))
        c = rs.uniform(-2, 2, size=(n, H)) if rep else np.zeros((n, H))
        comm = rs.randint(0, 2, size=n) if rep != 1 else np.zeros(n, dtype=np.int64)
        alive = (rs.randint(0, 2, size=n).astype(np.float64) if rep != 2 else np.eye(1, n)[0]) if use_alive else None
        info = {}
        if args.hard_attn:
            info["comm_action"] = comm
        if alive is not None:
            info["alive_mask"] = alive.copy()
        x_in = [torch.from_numpy(obs[None]), (torch.from_numpy(h), torch.from_numpy(c))]
        with torch.no_grad():
            act, val, (h2, c2) = net(x_in, info)
        lo, ov, oh2, oc2, ox = policy.forward(policy.params_to_f64(sd), obs, h, c,
                                              comm if args.hard_attn else None, alive, bool(args.hard_attn),
                                              args.comm_mode, args.comm_mask_zero)
        assert np.allclose(val.numpy()[:, 0], ov, rtol=1e-12, atol=1e-13), name
        assert np.allclose(h2.numpy(), oh2, rtol=1e-12, atol=1e-13), name
        assert np.allclose(c2.numpy(), oc2, rtol=1e-12, atol=1e-13), name
        for k in range(len(heads)):
            assert np.allclose(act[k].numpy()[0], lo[k], rtol=1e-12, atol=1e-13), name
            out["logp%d" % k].append(act[k].numpy()[0])
        out["obs"].append(obs); out["h"].append(h); out["c"].append(c); out["comm"].append(comm)
        out["alive"].append(np.ones(n) if alive is None else alive)
        out["value"].append(val.numpy()[:, 0]); out["h2"].append(h2.numpy()); out["c2"].append(c2.numpy())
        out["x"].append(ox)
    meta = dict(kind="forward", weights_seed=seed, obs_dim=obs_dim, heads=list(heads), use_alive=bool(use_alive),
                hard_attn=bool(args.hard_attn), comm_mode=args.comm_mode, comm_mask_zero=bool(args.comm_mask_zero),
                nagents=n, hid_size=H, comm_init=args.comm_init)
    save(name, meta, **{k: np.array(v) for k, v in out.items()})


# --------------------------------------------------------------------------
# 4. whole episodes through the reference's own Trainer.get_episode
# --------------------------------------------------------------------------
def gen_episode_case(name, seed, env_ids, wseed, hsteps=(0, 1), epoch=0, **kw):
    import torch
    torch.set_default_dtype(torch.float64)
    ref_shims.install()
    from comm import CommNetMLP
    from trainer import Trainer
    args = ref_shims.make_args(**kw)
    w = ref_shims.make_ref_env(args)
    ref_shims.finish_args(args, w)
    heads = args.naction_heads
    net = CommNetMLP(args, args.num_inputs)
    sd = make_weights(wseed, args.num_inputs, args.hid_size, heads, args.comm_init)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    params = policy.params_to_f64(sd)
    tr = Trainer(args, net, w)
    is_tj = args.env_name == "traffic_junction"
    tables = tj_tables_from_ref(w.env) if is_tj else None
    n, H, T = args.nagents, args.hid_size, args.max_steps
    eps = []
    for env_id in env_ids:
        rr = RefRandom(seed, env_id)
        hid = []
        orig_forward = net.forward

        def fwd(x, info={}, _o=orig_forward, _hid=hid):
            out = _o(x, info)
            _hid.append((out[2][0].detach().numpy().copy(), out[2][1].detach().numpy().copy()))
            return out
        net.forward = fwd
        orig_step = w.step

        def step(action, _o=orig_step, _rr=rr):
            _rr.group = -1
            out = _o(action)
            _rr.tick += 1
            _rr.head = 0
            return out
        w.step = step
        with routed(rr):
            episode, stat = tr.get_episode(epoch)
        net.forward, w.step = orig_forward, orig_step
        L = len(episode)
        # ---- oracle replay of trainer.py:26-126 with the same Philox streams ----
        orc = make_oracle_env(args, tables)
        if is_tj:
            oobs = orc.reset(epoch)
        else:
            oobs = orc.flat_obs(orc.reset(seed=seed, env_id=env_id, episode=0))
        oh, oc = np.zeros((n, H)), np.zeros((n, H))
        comm, alive = np.zeros(n, dtype=np.int64), None
        rec = dict(act=[], reward=[], value=[], alive=[], mini=[], emask=[], margin=[], comm_in=[], loc=[])
        for k in range(len(heads)):
            rec["logp%d" % k] = []
        hsel, csel = [], []
        for t in range(L):
            tr_t = episode[t]
            assert np.array_equal(tr_t.state.numpy()[0], oobs), "%s: state t=%d" % (name, t)
            lo, ov, oh, oc, _ = policy.forward(params, oobs, oh, oc, comm if args.hard_attn else None, alive,
                                               bool(args.hard_attn), args.comm_mode, args.comm_mask_zero)
            assert np.allclose(hid[t][0], oh, rtol=1e-11, atol=1e-12), "%s: h t=%d" % (name, t)
            assert np.allclose(tr_t.value.detach().numpy()[:, 0], ov, rtol=1e-11, atol=1e-12)
            a, margin = policy.sample_actions(lo, policy.action_draws(seed, env_id, t, n, len(heads)))
            ref_a = np.stack([np.asarray(x) for x in tr_t.action], 1)
            assert np.array_equal(a, ref_a), "%s: action t=%d" % (name, t)
            if is_tj:
                oobs, orew, odone, oinfo = orc.step(a[:, 0], seed=seed, env_id=env_id)
                alive = oinfo["alive_mask"]
                loc = orc.car_loc.copy()
            else:
                o, orew, odone, oinfo = orc.step(a[:, 0])
                oobs = orc.flat_obs(o)
                loc = np.vstack([orc.predator_loc, orc.prey_loc])
            if args.hard_attn:
                comm = a[:, -1] if not args.comm_action_one else np.ones(n, dtype=np.int64)
            rec["comm_in"].append(comm.copy())
            done = odone or t == T - 1
            last = t == L - 1
            assert done == last
            rew = orew + (orc.reward_terminal() if last else 0)
            assert np.array_equal(np.asarray(tr_t.reward), rew), "%s: reward t=%d" % (name, t)
            assert np.array_equal(tr_t.misc["alive_mask"], alive if alive is not None else np.ones(n))
            emask = np.zeros(n) if done else np.ones(n)
            mini = np.ones(n)
            if not done and is_tj:
                mini = 1 - oinfo["is_completed"]
            assert np.array_equal(tr_t.episode_mask, emask) and np.array_equal(tr_t.episode_mini_mask, mini)
            rec["act"].append(a); rec["reward"].append(rew); rec["value"].append(ov)
            rec["alive"].append(np.ones(n) if alive is None else alive.copy())
            rec["mini"].append(mini); rec["emask"].append(emask); rec["margin"].append(margin); rec["loc"].append(loc)
            for k in range(len(heads)):
                rec["logp%d" % k].append(lo[k])
            if t in hsteps or t == L - 1:
                hsel.append(oh.copy()); csel.append(oc.copy())
        ostat = dict(orc.stat)
        assert stat["num_steps"] == L
        assert stat.get("success") == ostat.get("success")
        nf = args.nfriendly                                   # trainer.py:73-75,86-88: friendly / enemy split
        assert np.allclose(stat["reward"], np.sum(rec["reward"], 0)[:nf])
        if getattr(args, "enemy_comm", False):
            assert np.allclose(stat["enemy_reward"], np.sum(rec["reward"], 0)[nf:])
        ep = {k: np.array(v) for k, v in rec.items()}
        ep["h_sel"], ep["c_sel"] = np.array(hsel), np.array(csel)
        ep["h_steps"] = np.array([t for t in range(L) if t in hsteps or t == L - 1])
        ep["success"] = np.array(int(stat.get("success", -1)))
        if "comm_action" in stat:
            ep["stat_comm"] = np.asarray(stat["comm_action"], dtype=np.float64)
        if "enemy_comm" in stat:
            ep["stat_enemy_comm"] = np.asarray(stat["enemy_comm"], dtype=np.float64)
            ep["stat_enemy_reward"] = np.asarray(stat["enemy_reward"], dtype=np.float64)
        eps.append(ep)
    meta = dict(kind="episode", seed=seed, env_ids=list(env_ids), weights_seed=wseed, epoch=epoch,
                args={k: v for k, v in vars(args).items() if isinstance(v, (int, float, str, bool))},
                obs_dim=int(args.num_inputs), heads=list(map(int, heads)))
    arrays = {}
    for i, ep in enumerate(eps):
        for k, v in ep.items():
            arrays["e%d_%s" % (i, k)] = v
    if is_tj:
        arrays["grid"] = tables["grid"]
        arrays["route_len"], arrays["route_cells"] = pack_routes(tables["routes"])
    save(name, meta, **arrays)


# --------------------------------------------------------------------------
# 5. REINFORCE gradient of a whole batch through the reference's Trainer.run_batch + compute_grad
# --------------------------------------------------------------------------
def gen_grad_case(name, seed, env_id, wseed, **kw):
    meta, arrays = ref_grad_case(seed, env_id, wseed, **kw)
    save(name, meta, **arrays)


def ref_grad_case(seed, env_id, wseed, full_grads=False, **kw):
    """(meta, arrays) of one reference worker's run_batch + compute_grad, checked against oracle/grad.py.  Gradients
    larger than 4096 values are stored as a sample + sums unless ``full_grads``."""
    import torch
    from . import grad as ograd
    from .rollout import run_episode
    torch.set_default_dtype(torch.float64)
    ref_shims.install()
    from comm import CommNetMLP
    from trainer import Trainer
    args = ref_shims.make_args(**kw)
    w = ref_shims.make_ref_env(args)
    ref_shims.finish_args(args, w)
    heads = args.naction_heads
    net = CommNetMLP(args, args.num_inputs)
    sd = make_weights(wseed, args.num_inputs, args.hid_size, heads, args.comm_init)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    tr = Trainer(args, net, w)
    is_tj = args.env_name == "traffic_junction"
    tables = tj_tables_from_ref(w.env) if is_tj else None
    rr = RefRandom(seed, env_id)
    orig_step, orig_reset = w.step, w.reset

    def step(action, _o=orig_step):
        rr.group = -1
        out = _o(action)
        rr.tick += 1
        rr.head = 0
        return out

    def reset(epoch, _o=orig_reset):
        out = _o(epoch)
        rr.episode += 1
        return out
    w.step, w.reset = step, reset
    with routed(rr):
        batch, stat = tr.run_batch(0)
    w.step, w.reset = orig_step, orig_reset
    tr.optimizer.zero_grad()
    s = tr.compute_grad(batch)
    ref_grads = {k: (v.grad.numpy().copy() if v.grad is not None else None) for k, v in net.named_parameters()}
    # ---- oracle replay ----
    params = policy.params_to_f64(sd)
    orc = make_oracle_env(args, tables)
    eps, tick, k = [], 0, 0
    while tick < stat["num_steps"]:
        ep = run_episode(orc, params, args, seed, env_id, epoch=0, tick0=tick, episode=k)
        eps.append(ep)
        tick += ep["num_steps"]
        k += 1
    assert tick == stat["num_steps"] and k == stat["num_episodes"]
    g, ostat, extra = ograd.compute_grad(params, eps, args)
    assert np.isclose(ostat["action_loss"], s["action_loss"], rtol=1e-9, atol=1e-9), (ostat, s)
    assert np.isclose(ostat["value_loss"], s["value_loss"], rtol=1e-9, atol=1e-9)
    assert np.isclose(ostat["entropy"], s["entropy"], rtol=1e-9, atol=1e-9)
    arrays = {}
    for key, rg in ref_grads.items():
        if rg is None:
            assert g[key] is None or not np.any(g[key]), key
            continue
        scale = max(1.0, float(np.abs(rg).max()))
        assert np.allclose(g[key], rg, rtol=1e-8, atol=1e-9 * scale), (name, key, np.abs(g[key] - rg).max())
        if rg.size <= 4096 or full_grads:
            arrays["g_" + key] = rg
        else:
            arrays["gsum_" + key] = np.array([rg.sum(), np.abs(rg).sum(), (rg ** 2).sum()])
            arrays["gsample_" + key] = rg.ravel()[::max(1, rg.size // 2048)][:2048].copy()
    meta = dict(kind="grad", seed=seed, env_id=env_id, weights_seed=wseed,
                args={k_: v for k_, v in vars(args).items() if isinstance(v, (int, float, str, bool))},
                obs_dim=int(args.num_inputs), heads=list(map(int, heads)), num_steps=int(stat["num_steps"]),
                num_episodes=int(stat["num_episodes"]), action_loss=float(s["action_loss"]),
                value_loss=float(s["value_loss"]), entropy=float(s["entropy"]))
    arrays["returns"] = extra["returns"]
    if is_tj:
        arrays["grid"] = tables["grid"]
        arrays["route_len"], arrays["route_cells"] = pack_routes(tables["routes"])
    return meta, arrays


def gen_rmsprop_case(name, seed, nupdates=5, lr=0.001):
    """torch.optim.RMSprop (the module trainer.py:21-22 instantiates) in float64, driven like
    Trainer.train_batch (trainer.py:245-256): zero_grad, accumulate, grad /= num_steps, step."""
    import torch
    g = torch.Generator().manual_seed(seed)
    shapes = [(32, 19), (32,), (7, 32), (7,), (1, 32), (1,), (5, 5), (3,)]      # last two: never get a gradient
    live = [True] * 6 + [False, False]
    params = [torch.nn.Parameter(torch.randn(*s, generator=g, dtype=torch.float64) * 0.1) for s in shapes]
    opt = torch.optim.RMSprop(params, lr=lr, alpha=0.97, eps=1e-6)
    arrays = {}
    for i, p_ in enumerate(params):
        arrays["p0_%d" % i] = p_.detach().numpy().copy()
    steps = []
    for u in range(nupdates):
        opt.zero_grad()
        ns = int(torch.randint(200, 900, (1,), generator=g))
        steps.append(ns)
        for i, p_ in enumerate(params):
            if live[i]:
                scale = 10.0 ** float(torch.randint(-3, 3, (1,), generator=g))      # wide dynamic range
                p_.grad = torch.randn(*shapes[i], generator=g, dtype=torch.float64) * scale * ns
                arrays["g%d_%d" % (u, i)] = p_.grad.numpy().copy()
        for p_ in params:                                                          # trainer.py:251-253
            if p_._grad is not None:
                p_._grad.data /= ns
        opt.step()
        for i, p_ in enumerate(params):
            arrays["p%d_%d" % (u + 1, i)] = p_.detach().numpy().copy()
    for i, p_ in enumerate(params):
        if live[i]:
            arrays["v_%d" % i] = opt.state[p_]["square_avg"].numpy().copy()
    meta = dict(kind="rmsprop", lr=lr, alpha=0.97, eps=1e-6, nupdates=nupdates, num_steps=steps, live=live,
                shapes=[list(s) for s in shapes], torch=torch.__version__)
    save(name, meta, **arrays)


def gen_log_case(name="log_contract"):
    """Per-epoch log / print contract: outputs of the reference's own main.py statements (oracle/ref_log.py) for a
    fixed sequence of epoch stats -> tests/golden/log_contract.json."""
    import copy
    import json
    from . import ref_log
    rs = np.random.RandomState(11)

    def epoch(kind, n=4):
        ne, ns = int(rs.randint(1, 200)), int(rs.randint(50, 9000))
        st = dict(num_episodes=ne, num_steps=ns, reward=(rs.randn(n) * ne).tolist(), steps_taken=ns,
                  value_loss=float(rs.rand() * ns), action_loss=float(rs.randn() * ns), entropy=float(rs.rand() * ns))
        if kind in ("pp", "tj"):
            st["success"] = int(rs.randint(0, ne + 1))
            st["comm_action"] = rs.randint(0, ns, size=n).astype(np.float64).tolist()
        if kind == "tj":
            st["add_rate"] = 0.05 * ne
        if kind == "empty":
            st["num_episodes"] = 0
        return st
    epochs = [epoch(k) for k in ("pp", "tj", "plain", "empty", "tj", "pp")]
    log = ref_log.make_log()
    lines = []
    for st in epochs:
        st = {k: (np.asarray(v) if isinstance(v, list) else v) for k, v in copy.deepcopy(st).items()}
        lines.append(ref_log.epoch_update(log, st, 1.2345))
    conv = lambda x: x.tolist() if isinstance(x, np.ndarray) else (x.item() if isinstance(x, np.generic) else x)
    out = dict(epochs=epochs, lines=lines, log={k: [conv(x) for x in f.data] for k, f in log.items()})
    with open(os.path.join(GOLDEN, name + ".json"), "w") as f:
        json.dump(out, f, indent=0)


def _load_path(modname, path):
    import importlib.util
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _test_cases(name):
    """A module of tests/, loaded by path: the cases a fixture is recorded for are defined once, in the test."""
    return _load_path("_cases_" + name, os.path.join(os.path.dirname(GOLDEN), name + ".py"))


def _write_json(name, out):
    path = os.path.join(GOLDEN, name + ".json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0)
    print("wrote %-40s %7.1f KB" % (name + ".json", os.path.getsize(path) / 1024.0))


def gen_host_logic_case(name="host_logic"):
    """What the reference's merge_stat (utils.py:15-29), parse_action_args (action_utils.py:5-25) and GymWrapper
    properties (env_wrappers.py:21-50) return for the cases of tests/test_host_logic.py -> tests/golden/host_logic.json."""
    import copy
    t = _test_cases("test_host_logic")
    ref_shims.install()
    import gym.spaces as gspaces                      # the stub installed by ref_shims
    ref = {m: _load_path("_ref_" + m, os.path.join(ref_shims.REF_ROOT, m + ".py"))
           for m in ("utils", "action_utils", "env_wrappers")}
    merged = []
    for src, dest in t.STAT_CASES:
        d = copy.deepcopy(dest)
        ref["utils"].merge_stat(copy.deepcopy(src), d)
        merged.append({k: t.typed(v) for k, v in d.items()})
    actions = [t._run(ref["action_utils"].parse_action_args, kw) for kw in t.ACTION_CASES]
    wrapper = {}
    for kind in ("pp", "tj", "multi"):
        w = ref["env_wrappers"].GymWrapper(t._FakeEnv(gspaces, kind))
        wrapper[kind] = [int(w.observation_dim), int(w.num_actions), int(w.dim_actions)]
    _write_json(name, dict(merge_stat=merged, parse_action_args=actions, gym_wrapper=wrapper))


def gen_log_main_py_case(name="log_main_py"):
    """The reference's log table (main.py:190-201: keys, plot flags, x axes, divisors) and what its main.py statements
    (oracle/ref_log.py) log and print for the epochs of tests/test_log_contract.py -> tests/golden/log_main_py.json."""
    import copy
    from . import ref_log
    t = _test_cases("test_log_contract")
    log = ref_log.make_log()
    lines = [ref_log.epoch_update(log, copy.deepcopy(st), 1.2345) for st in t.main_py_epochs()]
    _write_json(name, dict(keys=list(log.keys()), fields={k: [f.plot, f.x_axis, f.divide_by] for k, f in log.items()},
                           log={k: [t.to_jsonable(x) for x in f.data] for k, f in log.items()}, lines=lines))


def gen_apa_case(name="apa_pp_ic3net"):
    """--advantages_per_action off and on (trainer.py:189-199): the reference's losses and gradients for both settings
    on the same episodes, each checked against oracle/grad.py (which has no such flag) before it is written."""
    kw = dict(env_name="predator_prey", nagents=3, dim=5, vision=1, max_steps=8, hid_size=16, ic3net=True,
              batch_size=16)
    meta, arrays = ref_grad_case(19, 0, 7, full_grads=True, advantages_per_action=False, **kw)
    meta_on, on = ref_grad_case(19, 0, 7, full_grads=True, advantages_per_action=True, **kw)
    meta["on"] = {k: meta_on[k] for k in ("action_loss", "value_loss", "entropy", "num_steps", "num_episodes")}
    arrays.update({"on_" + k: v for k, v in on.items() if k.startswith("g_")})
    save(name, meta, **arrays)


def gen_variant_case(name, seed, obs_dim, heads, model, nrep=4, use_alive=False, **kw):
    """Forward fixtures of the policy variants (SURVEY 8(f)-4) from the UNMODIFIED reference modules: CommNetMLP with
    comm_passes > 1 / share_weights / the non-recurrent tanh branch, and models.MLP / models.RNN.  The module's own
    (seeded) initial state_dict is stored with the inputs and outputs; the numpy restatement
    oracle.policy.forward_variant is asserted equal on the way."""
    import torch
    torch.set_default_dtype(torch.float64)
    ref_shims.install()
    import comm as ref_comm
    import models as ref_models
    args = ref_shims.make_args(**kw)
    args.naction_heads, args.continuous = list(heads), False
    args.num_actions, args.dim_actions = list(heads), len(heads)
    torch.manual_seed(seed)
    if model == "commnet":
        if args.recurrent:
            args.rnn_type = "LSTM"
        net = ref_comm.CommNetMLP(args, obs_dim)
    elif model == "mlp":
        net = ref_models.MLP(args, obs_dim)
    else:
        net = ref_models.RNN(args, obs_dim)
    sd = {k: v.detach().numpy().copy() for k, v in net.state_dict().items()}
    params = policy.params_to_f64(sd)
    n, H = args.nagents, args.hid_size
    lstm = (model == "commnet" and args.recurrent) or (model == "rnn" and args.rnn_type == "LSTM")
    carries = (model == "rnn") or (model == "commnet" and args.recurrent)
    passes = args.comm_passes if model == "commnet" else 1
    roles = policy.roles_of(params, "commnet" if model == "commnet" else model, bool(args.recurrent), passes)
    variant = dict(passes=passes, x_tanh=(model == "mlp") or (model == "commnet" and not args.recurrent),
                   h_from_x=(model == "mlp") or (model == "commnet" and not args.recurrent))
    hard = bool(args.hard_attn) and model == "commnet"
    rs = np.random.RandomState(seed + 1)
    out = dict(obs=[], h=[], c=[], comm=[], alive=[], value=[], h2=[], c2=[])
    for k in range(len(heads)):
        out["logp%d" % k] = []
    for rep in range(nrep):
        obs = np.zeros((n, obs_dim))
        nz = rs.randint(0, obs_dim, size=(n, min(8, obs_dim)))
        for i in range(n):
            obs[i, nz[i]] = rs.randint(1, 4, size=nz.shape[1])
        h = rs.uniform(-1, 1, size=(n, H)) if rep else np.zeros((n, H))
        c = rs.uniform(-2, 2, size=(n, H)) if rep else np.zeros((n, H))
        comm = rs.randint(0, 2, size=n) if rep != 1 else np.zeros(n, dtype=np.int64)
        alive = rs.randint(0, 2, size=n).astype(np.float64) if (use_alive and model == "commnet") else None
        info = {}
        if hard:
            info["comm_action"] = comm
        if alive is not None:
            info["alive_mask"] = alive.copy()
        tobs = torch.from_numpy(obs[None])
        with torch.no_grad():
            if not carries:
                act, val = net(tobs, info)
                h2 = c2 = None
            elif lstm:
                act, val, (h2, c2) = net([tobs, (torch.from_numpy(h), torch.from_numpy(c))], info)
            else:
                act, val, h2 = net([tobs, torch.from_numpy(h[None])], info)
                c2 = None
        lo, ov, oh2, oc2 = policy.forward_variant(roles, obs, h if carries else None, c if lstm else None,
                                                  comm if hard else None, alive, hard, args.comm_mode,
                                                  bool(args.comm_mask_zero) or model != "commnet", **variant)
        assert np.allclose(val.numpy().reshape(-1), ov, rtol=1e-12, atol=1e-13), name
        for k in range(len(heads)):
            assert np.allclose(act[k].numpy().reshape(n, -1), lo[k], rtol=1e-12, atol=1e-13), name
            out["logp%d" % k].append(lo[k])
        if h2 is not None:
            assert np.allclose(h2.numpy().reshape(n, H), oh2, rtol=1e-12, atol=1e-13), name
        if c2 is not None:
            assert np.allclose(c2.numpy(), oc2, rtol=1e-12, atol=1e-13), name
        out["obs"].append(obs); out["h"].append(h); out["c"].append(c); out["comm"].append(comm)
        out["alive"].append(np.ones(n) if alive is None else alive)
        out["value"].append(ov); out["h2"].append(oh2); out["c2"].append(oc2 if oc2 is not None else np.zeros((n, H)))
    meta = dict(kind="variant", model=model, obs_dim=obs_dim, heads=list(heads), use_alive=bool(alive is not None),
                hard_attn=hard, lstm=bool(lstm), carries=bool(carries),
                args={k: v for k, v in vars(args).items() if isinstance(v, (int, float, str, bool))})
    arrays = {k: np.array(v) for k, v in out.items()}
    for k, v in sd.items():
        arrays["sd_" + k] = v
    save(name, meta, **arrays)


def gen_variant_cases():
    gen_variant_case("var_commnet_passes2", 91, 45, (5, 2), "commnet", nagents=5, hid_size=128, ic3net=True,
                     comm_passes=2, use_alive=True)
    gen_variant_case("var_commnet_share3", 92, 45, (5,), "commnet", nagents=4, hid_size=64, commnet=True,
                     comm_passes=3, share_weights=True)
    gen_variant_case("var_commnet_share3_h128", 98, 45, (5,), "commnet", nagents=5, hid_size=128, commnet=True,
                     comm_passes=3, share_weights=True, comm_mode="sum")
    gen_variant_case("var_commnet_passes4_h128", 99, 61, (2, 2), "commnet", nagents=7, hid_size=128, ic3net=True,
                     comm_passes=4, use_alive=True)
    gen_variant_case("var_commnet_nonrec2", 93, 61, (2, 2), "commnet", nagents=6, hid_size=128, ic3net=True,
                     recurrent=False, comm_passes=2, use_alive=True)
    gen_variant_case("var_commnet_nonrec_share", 94, 29, (5,), "commnet", nagents=3, hid_size=32, commnet=True,
                     recurrent=False, comm_passes=2, share_weights=True, comm_mode="sum")
    gen_variant_case("var_mlp", 95, 29, (5,), "mlp", nagents=3, hid_size=128, commnet=False, recurrent=False)
    gen_variant_case("var_rnn_tanh", 96, 29, (5,), "rnn", nagents=3, hid_size=128, commnet=False, recurrent=True,
                     rnn_type="MLP")
    gen_variant_case("var_rnn_lstm", 97, 61, (2,), "rnn", nagents=5, hid_size=128, commnet=False, recurrent=True,
                     rnn_type="LSTM")


def gen_enemy_comm_cases():
    """--enemy_comm (predator_prey_env.py:203-207,255,276-281; main.py:124-131; trainer.py:73-75,86-88,120-121): the prey
    is one more agent of the policy -- observation row, reward entry, communication; its action is ignored."""
    gen_env_case("env_pp_enemy", 30, 16, 4, env_name="predator_prey", nagents=3, dim=4, vision=1, enemy_comm=True)
    gen_env_case("env_pp_enemy_coop", 30, 17, 6, env_name="predator_prey", nagents=2, dim=3, vision=0, enemy_comm=True,
                 mode="cooperative")
    gen_episode_case("ep_pp_enemy_ic3net", 48, (0, 3), 58, hsteps=(0, 1, 8), env_name="predator_prey", nagents=3,
                     dim=5, vision=1, max_steps=20, hid_size=128, ic3net=True, enemy_comm=True)
    gen_grad_case("grad_pp_enemy_ic3net_h128", 68, 5, 78, env_name="predator_prey", nagents=3, dim=5, vision=1,
                  max_steps=12, hid_size=128, ic3net=True, enemy_comm=True, batch_size=40, detach_gap=5)
    # plain CommNet (everybody talks, the prey included), cooperative rewards, entropy bonus, normalised advantages
    gen_episode_case("ep_pp_enemy_commnet_coop", 49, (1,), 59, hsteps=(0, 1, 6), env_name="predator_prey", nagents=4,
                     dim=4, vision=0, max_steps=15, hid_size=128, commnet=True, enemy_comm=True, mode="cooperative")
    gen_grad_case("grad_pp_enemy_commnet_entr_h128", 69, 2, 79, env_name="predator_prey", nagents=4, dim=4, vision=0,
                  max_steps=10, hid_size=128, commnet=True, enemy_comm=True, mode="cooperative", batch_size=30,
                  entr=0.01, mean_ratio=1.0, gamma=0.9, normalize_rewards=True)


def gen_baseline_geometry_grad_cases():
    """Gradient fixtures at the GEOMETRY of the BASELINE configs c2 (predator-prey hard: 10 agents, dim 20, vision 1,
    O = 3636) and c5 (traffic junction hard: 20 cars, dim 18, 56 routes) -- shorter episodes, one env."""
    gen_grad_case("grad_pp_hard_ic3net_h128", 70, 6, 80, env_name="predator_prey", nagents=10, dim=20, vision=1,
                  max_steps=20, hid_size=128, ic3net=True, batch_size=35, detach_gap=8)
    gen_grad_case("grad_tj_hard_ic3net_h128", 71, 3, 81, env_name="traffic_junction", nagents=20, dim=18, vision=0,
                  max_steps=25, hid_size=128, ic3net=True, difficulty="hard", add_rate_min=0.2, add_rate_max=0.2,
                  batch_size=40, detach_gap=10)


def gen_nostay_cases():
    """--no_stay (predator_prey_env.py:88-92): four actions, the policy's env head has four logits."""
    gen_env_case("env_pp_nostay", 25, 18, 2, env_name="predator_prey", nagents=3, dim=4, vision=1, no_stay=True)
    gen_episode_case("ep_pp_nostay_commnet", 50, (0, 2), 60, hsteps=(0, 1, 5), env_name="predator_prey", nagents=3,
                     dim=4, vision=1, max_steps=15, hid_size=128, commnet=True, no_stay=True)
    # competitive rewards under policy-driven actions (0.05 / n_on, no 'success' statistic: :264-266, :284)
    gen_episode_case("ep_pp_comp_ic3net", 51, (1, 4), 61, hsteps=(0, 1, 9), env_name="predator_prey", nagents=4,
                     dim=3, vision=1, max_steps=20, hid_size=128, ic3net=True, mode="competitive")


def gen_hid128_grad_cases():
    """Gradient fixtures at hid_size 128 (the shape the tensor-core rollout and the BPTT kernels run at) covering the
    loss / comm variants: entropy bonus, normalised advantages, cooperative returns, comm_mode sum, plain CommNet (no
    hard attention), vision-1 windows with count features, IC-style comm_mask_zero."""
    gen_grad_case("grad_pp_v1_commnet_entr_h128", 65, 3, 75, env_name="predator_prey", nagents=4, dim=6, vision=1,
                  max_steps=15, hid_size=128, commnet=True, batch_size=40, mode="cooperative", entr=0.01,
                  mean_ratio=1.0, gamma=0.95, normalize_rewards=True)
    gen_grad_case("grad_tj_easy_commnet_sum_h128", 66, 1, 76, env_name="traffic_junction", nagents=5, dim=6, vision=0,
                  max_steps=20, hid_size=128, commnet=True, comm_mode="sum", difficulty="easy", add_rate_min=0.3,
                  add_rate_max=0.3, batch_size=50, mean_ratio=0.5, gamma=0.9, entr=0.005)
    gen_grad_case("grad_tj_medium_v1_ic_h128", 67, 2, 77, env_name="traffic_junction", nagents=6, dim=14, vision=1,
                  max_steps=30, hid_size=128, ic3net=True, comm_mask_zero=True, difficulty="medium",
                  add_rate_min=0.25, add_rate_max=0.25, batch_size=45, detach_gap=7)


def main():
    if "--variants-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_variant_cases()
        return 0
    if "--baseline-grad-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_baseline_geometry_grad_cases()
        return 0
    if "--nostay-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_nostay_cases()
        return 0
    if "--enemy-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_enemy_comm_cases()
        return 0
    if "--grad128-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_hid128_grad_cases()
        return 0
    if "--log-only" in sys.argv:
        gen_log_case()
        return 0
    if "--host-only" in sys.argv:
        import warnings
        warnings.filterwarnings("ignore")
        gen_host_logic_case()
        gen_log_main_py_case()
        gen_apa_case()
        return 0
    if "--rmsprop-only" in sys.argv:          # needs torch only, not the reference checkout
        gen_rmsprop_case("rmsprop_ref", 81)
        return 0
    if not ref_shims.reference_available():
        print("reference not available; nothing generated")
        return 1
    import warnings
    warnings.filterwarnings("ignore")
    gen_tj_tables()
    # env-only
    gen_env_case("env_pp_easy", 20, 11, 0, env_name="predator_prey", nagents=3, dim=5, vision=0)
    gen_env_case("env_pp_v1", 30, 12, 3, env_name="predator_prey", nagents=2, dim=4, vision=1)
    gen_env_case("env_pp_coop", 30, 13, 1, env_name="predator_prey", nagents=4, dim=3, vision=1, mode="cooperative")
    gen_env_case("env_pp_comp", 30, 14, 2, env_name="predator_prey", nagents=4, dim=3, vision=2, mode="competitive")
    gen_env_case("env_pp_hard", 12, 15, 5, store_obs=False, env_name="predator_prey", nagents=10, dim=20, vision=1)
    gen_env_case("env_tj_easy", 40, 21, 0, env_name="traffic_junction", nagents=5, dim=6, vision=0,
                 difficulty="easy", add_rate_min=0.3, add_rate_max=0.3)
    gen_env_case("env_tj_medium", 60, 22, 1, env_name="traffic_junction", nagents=10, dim=14, vision=0,
                 difficulty="medium", add_rate_min=0.2, add_rate_max=0.2)
    gen_env_case("env_tj_medium_v1", 40, 23, 2, env_name="traffic_junction", nagents=10, dim=14, vision=1,
                 difficulty="medium", add_rate_min=0.3, add_rate_max=0.3)
    gen_env_case("env_tj_hard", 60, 24, 3, env_name="traffic_junction", nagents=20, dim=18, vision=0,
                 difficulty="hard", add_rate_min=0.2, add_rate_max=0.2)
    gen_env_case("env_tj_hard_v1", 30, 25, 4, store_obs=False, env_name="traffic_junction", nagents=20, dim=18,
                 vision=1, difficulty="hard", add_rate_min=0.25, add_rate_max=0.25)
    # forward
    gen_forward_case("fwd_ic3net_pp", 31, 29, (5, 2), False, nagents=3, hid_size=128, ic3net=True)
    gen_forward_case("fwd_ic3net_tj", 32, 61, (2, 2), True, nagents=10, hid_size=128, ic3net=True,
                     env_name="traffic_junction")
    gen_forward_case("fwd_commnet", 33, 45, (5,), False, nagents=5, hid_size=64, commnet=True)
    gen_forward_case("fwd_commnet_sum", 34, 45, (5,), True, nagents=5, hid_size=64, commnet=True, comm_mode="sum")
    gen_forward_case("fwd_ic_nocomm", 35, 29, (5, 2), False, nagents=3, hid_size=32, ic3net=True, comm_mask_zero=True)
    gen_forward_case("fwd_comm_zero_init", 36, 29, (5, 2), False, nagents=3, hid_size=32, ic3net=True, comm_init="zeros")
    # episodes
    gen_episode_case("ep_pp_easy_ic3net", 41, (0, 1, 2), 51, hsteps=(0, 1, 5, 10), env_name="predator_prey",
                     nagents=3, dim=5, vision=0, max_steps=20, hid_size=128, ic3net=True)
    gen_episode_case("ep_pp_hard_ic3net", 42, (7,), 52, hsteps=(0, 1, 40), env_name="predator_prey",
                     nagents=10, dim=20, vision=1, max_steps=80, hid_size=128, ic3net=True)
    gen_episode_case("ep_pp_hard_commnet", 43, (3,), 53, hsteps=(0, 1, 40), env_name="predator_prey",
                     nagents=10, dim=20, vision=1, max_steps=80, hid_size=128, commnet=True)
    gen_episode_case("ep_tj_easy_ic3net", 44, (0, 1), 54, hsteps=(0, 1, 10), env_name="traffic_junction",
                     nagents=5, dim=6, vision=0, max_steps=20, hid_size=128, ic3net=True, difficulty="easy",
                     add_rate_min=0.3, add_rate_max=0.3)
    gen_episode_case("ep_tj_medium_ic3net", 45, (0, 5), 55, hsteps=(0, 1, 20), env_name="traffic_junction",
                     nagents=10, dim=14, vision=0, max_steps=40, hid_size=128, ic3net=True, difficulty="medium",
                     add_rate_min=0.05, add_rate_max=0.02)
    gen_episode_case("ep_tj_hard_ic3net", 46, (2,), 56, hsteps=(0, 1, 40), epoch=300, env_name="traffic_junction",
                     nagents=20, dim=18, vision=0, max_steps=80, hid_size=128, ic3net=True, difficulty="hard",
                     add_rate_min=0.02, add_rate_max=0.05, curr_start=250, curr_end=1250)
    gen_episode_case("ep_tj_medium_v1_commnet", 47, (1,), 57, hsteps=(0, 1, 20), env_name="traffic_junction",
                     nagents=10, dim=14, vision=1, max_steps=40, hid_size=64, commnet=True, difficulty="medium",
                     add_rate_min=0.2, add_rate_max=0.2)
    gen_grad_case("grad_pp_easy_ic3net", 61, 2, 71, env_name="predator_prey", nagents=3, dim=5, vision=0,
                  max_steps=20, hid_size=128, ic3net=True, batch_size=50, detach_gap=10, value_coeff=0.01)
    gen_grad_case("grad_pp_coop_commnet_entr", 62, 1, 72, env_name="predator_prey", nagents=4, dim=3, vision=1,
                  max_steps=12, hid_size=32, commnet=True, batch_size=40, mode="cooperative", entr=0.01,
                  mean_ratio=1.0, gamma=0.95, normalize_rewards=True)
    gen_grad_case("grad_tj_medium_ic3net", 63, 4, 73, env_name="traffic_junction", nagents=10, dim=14, vision=0,
                  max_steps=40, hid_size=128, ic3net=True, difficulty="medium", add_rate_min=0.2, add_rate_max=0.2,
                  batch_size=70, detach_gap=10)
    gen_grad_case("grad_tj_easy_commnet", 64, 0, 74, env_name="traffic_junction", nagents=5, dim=6, vision=0,
                  max_steps=20, hid_size=64, commnet=True, difficulty="easy", add_rate_min=0.3, add_rate_max=0.3,
                  batch_size=50, mean_ratio=0.5, gamma=0.9)
    gen_hid128_grad_cases()
    gen_enemy_comm_cases()
    gen_nostay_cases()
    gen_baseline_geometry_grad_cases()
    gen_variant_cases()
    gen_rmsprop_case("rmsprop_ref", 81)
    gen_log_case()
    gen_host_logic_case()
    gen_log_main_py_case()
    gen_apa_case()
    return 0


if __name__ == "__main__":
    sys.exit(main())
