"""CPU tests of the host-side glue the rollout's callers rely on: merge_stat (utils.py:15-29) and
parse_action_args (action_utils.py:5-25) -- fixed expectations, plus a differential check against what the reference's
own functions return for the same cases (tests/golden/host_logic.json, recorded by oracle/gen_golden.py)."""
import argparse
import copy
import json
import os

import numpy as np
import pytest

from ic3net_b200.action_utils import parse_action_args
from ic3net_b200.utils import merge_stat

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _golden(name):
    with open(os.path.join(GOLDEN, name + ".json")) as f:
        return json.load(f)


STAT_CASES = [
    (dict(a=1, b=2.5), dict()),
    (dict(a=1, r=np.array([1.0, 2.0])), dict(a=4, r=np.array([0.5, 0.5]))),
    (dict(s="x"), dict(s="y")),
    (dict(s="x"), dict(s=["y"])),
    (dict(s=["x", "z"]), dict(s=["y"])),
    (dict(s=["x"]), dict(s="y")),
    (dict(n=3, new=np.zeros(2)), dict(n=np.array([1, 1]))),
    (dict(flag=True), dict(flag=2)),
]


def typed(x):
    """JSON form of a merged value that keeps its type apart (bool / int / float / str, ndarray dtype, nesting)."""
    if isinstance(x, np.ndarray):
        return ["ndarray", str(x.dtype), x.tolist()]
    if isinstance(x, list):
        return ["list", [typed(v) for v in x]]
    if isinstance(x, np.generic):
        return [type(x).__name__, x.item()]
    return [type(x).__name__, x]


def test_merge_stat_rules():
    d = dict(a=4, r=np.array([0.5, 0.5]))
    merge_stat(dict(a=1, r=np.array([1.0, 2.0]), new="v"), d)
    assert d["a"] == 5 and np.array_equal(d["r"], [1.5, 2.5]) and d["new"] == "v"
    d = dict(s="y")
    merge_stat(dict(s="x"), d)
    assert d["s"] == ["y", "x"]
    merge_stat(dict(s="z"), d)
    assert d["s"] == ["y", "x", "z"]
    merge_stat(dict(s=["p", "q"]), d)
    assert d["s"] == ["y", "x", "z", "p", "q"]
    d = dict(s="y")
    merge_stat(dict(s=["x"]), d)
    assert d["s"] == ["y", ["x"]]                       # a list merged into a plain value nests (reference quirk)


@pytest.mark.parametrize("case", range(len(STAT_CASES)))
def test_merge_stat_matches_reference(case):
    src, dest = STAT_CASES[case]
    d = copy.deepcopy(dest)
    merge_stat(copy.deepcopy(src), d)
    ours = json.loads(json.dumps({k: typed(v) for k, v in d.items()}))
    assert ours == _golden("host_logic")["merge_stat"][case]


ACTION_CASES = [
    dict(num_actions=[5], dim_actions=1, nactions="1"),
    dict(num_actions=[5, 2], dim_actions=2, nactions="1"),
    dict(num_actions=[2, 2], dim_actions=1, nactions="1"),
    dict(num_actions=[0], dim_actions=1, nactions="1"),
    dict(num_actions=[0], dim_actions=3, nactions="4"),
    dict(num_actions=[-1], dim_actions=2, nactions="3:5"),
    dict(num_actions=[0], dim_actions=1, nactions="0"),
    dict(num_actions=[0], dim_actions=1, nactions=""),
]


def _run(fn, kw):
    a = argparse.Namespace(**copy.deepcopy(kw))
    try:
        fn(a)
    except Exception as e:                               # noqa: BLE001 - the exception type is part of the behaviour
        return type(e).__name__, None
    return None, (getattr(a, "continuous", None), getattr(a, "naction_heads", None))


def test_parse_action_args_rules():
    assert _run(parse_action_args, ACTION_CASES[0]) == (None, (False, [5]))
    assert _run(parse_action_args, ACTION_CASES[1]) == (None, (False, [5, 2]))
    assert _run(parse_action_args, ACTION_CASES[2]) == (None, (False, [2]))
    assert _run(parse_action_args, ACTION_CASES[3]) == (None, (True, None))
    assert _run(parse_action_args, ACTION_CASES[4]) == (None, (False, [4, 4, 4]))
    assert _run(parse_action_args, ACTION_CASES[5]) == (None, (False, [3, 5]))
    assert _run(parse_action_args, ACTION_CASES[6])[0] == "RuntimeError"
    assert _run(parse_action_args, ACTION_CASES[7])[0] == "ValueError"


@pytest.mark.parametrize("case", range(len(ACTION_CASES)))
def test_parse_action_args_matches_reference(case):
    ours = json.loads(json.dumps(_run(parse_action_args, ACTION_CASES[case])))
    assert ours == _golden("host_logic")["parse_action_args"][case]


# ---- GymWrapper on duck-typed environments (no GPU needed) ---------------------------------------------
class _FakeEnv(object):
    """Minimal batched env: records what the wrapper passes down."""

    def __init__(self, spaces_mod, kind, nenvs=3, nagents=4, takes_epoch=False):
        sp = spaces_mod
        self.nenvs, self.n = nenvs, nagents
        if kind == "pp":                                   # predator_prey_env.py:95,107
            self.observation_space = sp.Box(low=0, high=1, shape=(29, 3, 3), dtype=int)
            self.action_space = sp.MultiDiscrete([5])
        elif kind == "tj":                                 # traffic_junction_env.py:109,135-148
            self.observation_space = sp.Tuple((sp.Discrete(2), sp.Discrete(12), sp.MultiBinary((3, 3, 59))))
            self.action_space = sp.Discrete(2)
        else:                                              # two action dimensions reach the env
            self.observation_space = sp.Box(low=0, high=1, shape=(7,), dtype=int)
            self.action_space = sp.MultiDiscrete([4, 3])
        self.calls = []
        if takes_epoch:
            self.reset = lambda epoch=None: self._reset(epoch)
        else:
            self.reset = lambda: self._reset("none")
        self.stat = dict(success=1, steps_taken=9)

    def _obs(self, odim):
        import torch
        return torch.arange(self.nenvs * self.n * odim, dtype=torch.float32).reshape(self.nenvs, self.n, -1)

    def _reset(self, epoch):
        self.calls.append(("reset", epoch))
        return self._obs(self._odim)

    def step(self, action):
        self.calls.append(("step", action))
        return self._obs(self._odim), "r", "d", dict(k=1)

    def get_stat(self):
        return dict(self.stat)


@pytest.mark.parametrize("kind,odim,nact,dact", [("pp", 29 * 9, 5, 1), ("tj", 2 + 9 * 59, 2, 1), ("multi", 7, 4, 2)])
def test_gym_wrapper_surface(kind, odim, nact, dact):
    from ic3net_b200 import spaces
    from ic3net_b200.env_wrappers import GymWrapper
    env = _FakeEnv(spaces, kind, takes_epoch=(kind == "tj"))
    env._odim = odim
    w = GymWrapper(env)
    assert (w.observation_dim, w.num_actions, w.dim_actions, w.nenvs) == (odim, nact, dact, 3)
    assert w.action_space is env.action_space
    obs = w.reset(7)
    assert tuple(obs.shape) == (3, 4, odim)
    assert env.calls[-1] == ("reset", 7 if kind == "tj" else "none")        # epoch only where reset() takes it
    heads = ["head0", "head1"]
    o, r, d, info = w.step(heads)
    assert env.calls[-1] == ("step", "head0" if dact == 1 else heads)       # one action dim: only head 0 reaches the env
    assert tuple(o.shape) == (3, 4, odim) and (r, d, info) == ("r", "d", dict(k=1))
    assert w.get_stat() == dict(success=1) and env.stat["steps_taken"] == 9
    assert np.array_equal(w.reward_terminal(), np.zeros(1))                  # env without reward_terminal()
    env.reward_terminal = lambda: "rt"
    assert w.reward_terminal() == "rt"
    assert w._flatten_obs(obs).shape == obs.shape


@pytest.mark.parametrize("kind", ["pp", "tj", "multi"])
def test_gym_wrapper_matches_reference_properties(kind):
    """observation_dim / num_actions / dim_actions against the reference's GymWrapper on the same space objects (the
    gym space stand-ins of oracle/ref_shims.py, which the reference ran on when the fixture was recorded)."""
    from ic3net_b200.env_wrappers import GymWrapper
    from oracle.ref_shims import _make_gym_stub
    a = GymWrapper(_FakeEnv(_make_gym_stub()["gym.spaces"], kind))
    assert [a.observation_dim, a.num_actions, a.dim_actions] == _golden("host_logic")["gym_wrapper"][kind]


def test_enemy_comm_derived_args_and_stat_split():
    """--enemy_comm host logic (main.py:124-131; trainer.py:73-75,86-88,120-121): the prey joins the agents of the policy,
    and its reward / gate sums are reported under their own keys.  CPU only: derive_args and the host half of
    Trainer.stat_from_vector."""
    from types import SimpleNamespace
    from ic3net_b200 import main as cli
    from ic3net_b200.trainer import Trainer
    a = cli.derive_args(argparse.Namespace(ic3net=True, env_name="predator_prey", nagents=3, nenemies=1, enemy_comm=True,
                                           plot=False, display=False, commnet=False, hard_attn=False, mean_ratio=1.0))
    assert (a.nfriendly, a.nagents) == (3, 4) and a.commnet and a.hard_attn and a.mean_ratio == 0
    with pytest.raises(RuntimeError):          # main.py:129-130
        cli.derive_args(argparse.Namespace(ic3net=False, env_name="predator_prey", nagents=3, enemy_comm=True, plot=False,
                                           display=False))
    # stat vector layout: [episodes, steps, success, flags, reward[N], comm_action[N]] with N = 4 agent rows
    v = np.array([5, 40, 2, 0, -1.0, -2.0, -3.0, 1.5, 7, 8, 9, 4], dtype=np.float64)
    fake = SimpleNamespace(args=a, is_tj=False)
    a.mode = "mixed"
    st = Trainer.stat_from_vector(fake, v)
    assert st["num_episodes"] == 5 and st["num_steps"] == 40 and st["steps_taken"] == 40 and st["success"] == 2
    assert np.array_equal(st["reward"], [-1.0, -2.0, -3.0]) and np.array_equal(st["enemy_reward"], [1.5])
    assert np.array_equal(st["comm_action"], [7, 8, 9]) and np.array_equal(st["enemy_comm"], [4])
    b = argparse.Namespace(**{**vars(a), "enemy_comm": False, "nfriendly": 4})
    st = Trainer.stat_from_vector(SimpleNamespace(args=b, is_tj=False), v)
    assert len(st["reward"]) == 4 and "enemy_reward" not in st and "enemy_comm" not in st
    v[3] = 0x10
    with pytest.raises(RuntimeError):          # a device-side error flag is never swallowed
        Trainer.stat_from_vector(fake, v)


def test_advantages_per_action_is_the_same_loss_in_the_reference():
    """--advantages_per_action (trainer.py:189-199) multiplies the advantage into every head's log-probability before the
    sum instead of after it: the loss -- and therefore the gradient -- is the same number.  This repo accepts the flag and
    has one code path.  The fixture holds the unmodified reference's losses and gradients with the flag off and on, on
    the same episodes: they agree, and the float64 oracle (oracle/grad.py) reproduces both."""
    from helpers import load_golden, make_oracle_env, ns
    from oracle import grad as ograd
    from oracle import policy
    from oracle.gen_golden import make_weights
    from oracle.rollout import run_episode
    meta, z = load_golden("apa_pp_ic3net")
    assert not meta["args"]["advantages_per_action"]
    for k in ("action_loss", "value_loss", "entropy"):
        assert np.isclose(meta[k], meta["on"][k], rtol=1e-12, atol=1e-12), k
    args = ns(meta["args"])
    p = policy.params_to_f64(make_weights(meta["weights_seed"], meta["obs_dim"], args.hid_size, meta["heads"],
                                          args.comm_init))
    env = make_oracle_env(args)
    eps, tick = [], 0
    while tick < meta["num_steps"]:
        eps.append(run_episode(env, p, args, meta["seed"], meta["env_id"], epoch=0, tick0=tick, episode=len(eps)))
        tick += eps[-1]["num_steps"]
    assert len(eps) == meta["num_episodes"] == meta["on"]["num_episodes"]
    g, st, _ = ograd.compute_grad(p, eps, args)
    for k in ("action_loss", "value_loss", "entropy"):
        assert np.isclose(st[k], meta[k], rtol=1e-9, atol=1e-9), k
    keys = [k for k in z.files if k.startswith("g_")]
    assert len(keys) >= 8 and sorted("on_" + k for k in keys) == sorted(k for k in z.files if k.startswith("on_"))
    for key in keys:
        assert np.allclose(z[key], z["on_" + key], rtol=1e-10, atol=1e-12), key
        assert np.allclose(g[key[2:]], z[key], rtol=1e-8, atol=1e-10), key
