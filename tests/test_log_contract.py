"""SURVEY 8(f)-3: the stat / log pipeline the hot path's callers rely on.

(1) differential: ic3net_b200.main.update_log / epoch_lines against what the reference's own main.py statements
    (oracle/ref_log.py executes main.py:190-201,218-244 from the unmodified source text) logged and printed for
    randomised epoch stats, including fields an epoch did not produce and zero divisors (tests/golden/log_main_py.json);
(2) the same against a committed fixture of reference outputs (tests/golden/log_contract.json), so the contract is
    checked where the reference is absent;
(3) 1-rank vs 2-rank: statistics merged over ranks with the reference's merge rule give the same per-epoch values
    as one worker holding all the slots;
(4) checkpoint interchange of the `log` object (pickled as utils.LogField, main.py:260-272)."""
import copy
import json
import os
import sys

import numpy as np

from ic3net_b200 import main as m
from ic3net_b200.utils import LogField, merge_stat

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "log_contract.json")
GOLDEN_MAIN_PY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "log_main_py.json")


def random_epoch(rs, nagents, kind):
    ne, ns = int(rs.randint(1, 200)), int(rs.randint(50, 9000))
    st = dict(num_episodes=ne, num_steps=ns, reward=rs.randn(nagents) * ne, steps_taken=ns,
              value_loss=float(rs.rand() * ns), action_loss=float(rs.randn() * ns), entropy=float(rs.rand() * ns))
    if kind in ("pp", "tj"):
        st["success"] = int(rs.randint(0, ne + 1))
        st["comm_action"] = rs.randint(0, ns, size=nagents).astype(np.float64)
    if kind == "tj":
        st["add_rate"] = 0.05 * ne
    if kind == "empty":
        st["num_episodes"] = 0                     # divisor 0: fields stay un-normalised (main.py:223)
    return st


def to_jsonable(x):
    if isinstance(x, np.ndarray):
        return x.tolist()
    if isinstance(x, (np.floating, np.integer)):
        return x.item()
    return x


def run_ours(epochs):
    log = m.make_log()
    lines = []
    for st in epochs:
        st = copy.deepcopy(st)
        ep = m.update_log(log, st)
        lines.append(m.epoch_lines(ep, st, 1.2345))
    return {k: [to_jsonable(x) for x in v.data] for k, v in log.items()}, lines


def main_py_epochs():
    rs = np.random.RandomState(3)
    return [random_epoch(rs, 4, kind) for kind in ("pp", "tj", "plain", "empty", "tj", "pp")]


def test_update_log_matches_reference_main_py_text():
    with open(GOLDEN_MAIN_PY) as f:
        fx = json.load(f)
    ours, our_lines = run_ours(main_py_epochs())
    mine = m.make_log()
    assert list(mine.keys()) == fx["keys"]
    for k, f in mine.items():
        assert [f.plot, f.x_axis, f.divide_by] == fx["fields"][k], k
        assert json.dumps(fx["log"][k]) == json.dumps(ours[k]), k
    assert fx["lines"] == our_lines


def test_update_log_matches_committed_reference_fixture():
    fx = json.load(open(GOLDEN))
    epochs = [{k: (np.asarray(v) if isinstance(v, list) else v) for k, v in st.items()} for st in fx["epochs"]]
    ours, lines = run_ours(epochs)
    for k, series in fx["log"].items():
        assert json.dumps(series) == json.dumps(ours[k]), k
    assert fx["lines"] == lines


def test_two_ranks_merge_to_the_single_worker_epoch_values():
    rs = np.random.RandomState(5)
    r0, r1 = random_epoch(rs, 3, "tj"), random_epoch(rs, 3, "tj")
    both = dict()
    merge_stat(copy.deepcopy(r0), both)
    merge_stat(copy.deepcopy(r1), both)              # multi_processing.py:86-88
    from ic3net_b200.multi_gpu import pack_stat, unpack_stat
    import torch
    v0, shapes = pack_stat(r0, torch.device("cpu"))
    v1, _ = pack_stat(r1, torch.device("cpu"))
    reduced = unpack_stat(v0 + v1, shapes, {})       # what the all-reduce leaves on every rank
    a, la = run_ours([both])
    b, lb = run_ours([reduced])
    assert json.dumps(a) == json.dumps(b) and la == lb
    # add_rate: every episode reports the env's add_rate, so the epoch value is the rate itself
    assert abs(a["add_rate"][0] - 0.05) < 1e-12


def test_log_pickles_under_the_reference_module_name(tmp_path):
    import pickle
    import torch
    log = m.make_log()
    m.update_log(log, random_epoch(np.random.RandomState(0), 2, "pp"))
    path = str(tmp_path / "ck.pt")

    class FakeNet(object):
        def state_dict(self):
            return {}

        def load_state_dict(self, d):
            pass
    m.save_checkpoint(path, FakeNet(), log, FakeNet())
    blob = open(path, "rb").read()
    assert b"ic3net_b200" not in blob                # the reference can unpickle it: class path is utils.LogField
    assert b"utils" in blob and LogField.__module__ == "ic3net_b200.utils"     # alias removed again
    log2 = m.make_log()
    m.load_checkpoint(path, FakeNet(), log2, FakeNet())
    assert log2["reward"].data[0].tolist() == log["reward"].data[0].tolist() and isinstance(log2["reward"], LogField)
