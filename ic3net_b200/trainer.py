"""Batched GPU rollout + REINFORCE gradient behind the reference's ``trainer.Trainer`` surface
(trainer.py:14-262).

``Trainer(args, policy_net, env)`` drives ``env.nenvs`` independent environment slots in
lock-step on one GPU.  Each slot plays the role of one reference process: it runs episode after
episode (auto-reset, hidden state zeroed, nobody talks at t = 0), and ``run_batch`` follows the
reference's batch boundary (trainer.py:231-237): a slot plays WHOLE episodes until it holds
``>= batch_size`` steps -- its last episode overshoots -- and then halts (the lock-step loop runs
``batch_size + max_steps - 1`` iterations when episodes can end early, ``ceil(batch_size /
max_steps) * max_steps`` when they cannot; halted slots leave null records with ``valid = 0``).
``args.batch_boundary = 'cut'`` selects the round-1 behaviour instead (a fixed number of lock-steps,
episodes still open at the end are cut there).

Rollout (the hot path): one lock-step iteration is a handful of kernel launches and no host
synchronisation:
  encoder (index form from the env state, or obs-gather + dense encoder)
  -> policy step (comm mean, C, LSTM, heads, sampling; tcgen05 or fp32 SIMT kernels)
  -> env step + Trainer.get_episode bookkeeping + auto-reset (ic3_rollout_io).
The whole T-step sequence can be captured once into a CUDA graph (``use_graph``).

Gradient (``compute_grad``, trainer.py:128-225; scope row 8(f)-1): returns by a CUDA scan kernel,
then the policy forward is RECOMPUTED with differentiable torch ops (fp32, batched over all slots)
in windows of ``grad_window`` steps processed last-to-first; (h, c) at every window start are
checkpointed during the rollout and the gradient w.r.t. them is handed to the previous window,
so back-propagation through time is exact (truncated only where the reference truncates it:
``detach_gap``, trainer.py:56-60, and episode starts).
"""
import ctypes as C
import math
from collections import namedtuple

import torch
import torch.nn.functional as F

from . import _lib
from .optim import FlatRMSprop
from .utils import merge_stat

Transition = namedtuple('Transition', ('state', 'action', 'action_out', 'value', 'episode_mask',
                                       'episode_mini_mask', 'next_state', 'reward', 'misc'))

RolloutBatch = namedtuple('RolloutBatch', ('action', 'logp', 'value', 'reward', 'episode_mask',
                                           'episode_mini_mask', 'alive_mask', 'valid'))


def policy_forward_torch(net, x, h, c, g, n_alive):
    """Differentiable torch restatement of the policy step the kernels run (comm.py:134-244 for every variant of
    ic3_policy_cfg.cell / passes / x_tanh / h_from_x), on the module's own parameters.  x: encoder output [R, H];
    h, c: [R, H] entering the step; g: comm gate per agent [B, N] (alive * comm_action); n_alive: [B, 1].
    Returns (h', c', value [R, 1], [log-probs per head [R, na]])."""
    w, cp = net._kernel_weights(), net._cfg_proto
    B, N = g.shape
    H = x.shape[1]
    lstm = cp['cell'] == _lib.CELL_LSTM
    if cp['x_tanh']:
        x = torch.tanh(x)                                                              # comm.py:127-128
    hid = x if cp['h_from_x'] else h                                                   # comm.py:129
    den = torch.where(n_alive > 1, n_alive - 1, torch.ones_like(n_alive)) if cp['comm_avg'] else torch.ones_like(n_alive)
    gg = g.unsqueeze(-1)
    for ps in range(max(1, cp['passes'])):                                             # comm.py:179
        if cp['comm_mask_zero'] or N < 2:
            S = torch.zeros_like(hid)
        else:
            hv = hid.view(B, N, H)
            tot = (gg * hv).sum(1, keepdim=True)
            S = (gg * (tot - gg * hv) / den.unsqueeze(-1)).reshape(B * N, H)           # comm.py:181-205
        cvec = F.linear(S, w['c_w'][ps], w['c_b'][ps])                                 # comm.py:206
        if lstm:
            gates = F.linear(x + cvec, w['w_ih'], w['b_ih']) + F.linear(hid, w['w_hh'], w['b_hh'])   # comm.py:211-218
            gi, gf, gq, go = gates.chunk(4, dim=1)
            c = torch.sigmoid(gf) * c + torch.sigmoid(gi) * torch.tanh(gq)
            hid = torch.sigmoid(go) * torch.tanh(c)
        else:
            hid = torch.tanh(x + F.linear(hid, w['f_w'][ps], w['f_b'][ps]) + cvec)     # comm.py:220-224
    value = F.linear(hid, w['value_w'], w['value_b'])                                  # comm.py:228
    logps = [F.log_softmax(F.linear(hid, hw, hb), dim=-1) for hw, hb in zip(w['head_w'], w['head_b'])]
    return hid, c, value, logps


class Trainer(object):
    def __init__(self, args, policy_net, env):
        if not hasattr(policy_net, 'packed'):
            raise NotImplementedError("Trainer drives policies that run on the CUDA kernels (CommNetMLP, models.MLP, "
                                      "models.RNN); models.Random has no kernel path")
        self.args = args
        self.policy_net = policy_net
        self.env = env                       # GymWrapper
        self.display = False
        self.last_step = False
        # trainer.py:21-22 RMSprop(lr, alpha=0.97, eps=1e-6) as one kernel over flat buffers (optim.py)
        self.optimizer = FlatRMSprop(policy_net.parameters(), lr=args.lrate, alpha=0.97, eps=1e-6)
        self.params = [p for p in self.policy_net.parameters()]
        self.obs_mode = getattr(args, 'obs_mode', 'index')      # 'index' | 'dense'
        self.use_graph = bool(getattr(args, 'use_graph', False))
        self.is_tj = args.env_name == 'traffic_junction'
        self.record_for_grad = bool(getattr(args, 'record_for_grad', False))
        self.grad_window = int(getattr(args, 'grad_window', 40))
        # compute_grad implementation: 'kernels' = hand-written BPTT (csrc/bptt_tc.cu; tensor-core policy path, at most
        # 7 action logits, observation pattern of <= 512 columns), 'autograd' = windowed recompute under torch autograd,
        # 'manual' = explicit formulas with torch GEMMs (bptt.py).  Default: kernels when the configuration allows.
        self.grad_impl = getattr(args, 'grad_impl', None) or 'auto'
        self.grad_kernels = False
        self._bptt = None
        self._buf = None
        self._graph = None
        self._graph_key = None
        # encoder layout of this environment (class terms / counts summed separately, comm.py set_obs_layout) and
        # the per-position table of the class terms for the fused index encoder, rebuilt when the weights change
        policy_net.set_obs_layout(*getattr(env.env, 'obs_layout', (0, 0, 0)))
        self.use_xtable = bool(getattr(args, 'encoder_table', True))
        self._xtable = None
        self._xtable_key = None
        if self.record_for_grad and self.grad_impl in ('auto', 'kernels'):
            ok = self._bptt_supported()
            if self.grad_impl == 'kernels' and not ok:
                raise NotImplementedError("grad_impl='kernels' needs the tensor-core policy path (hid_size 128), the "
                                          "per-position encoder table, <= 7 action logits and a small vision window")
            self.grad_kernels = ok
        if self.grad_impl == 'auto':
            self.grad_impl = 'kernels' if self.grad_kernels else 'autograd'

    def _bptt_supported(self):
        e, net = self.env.env, self.policy_net
        W = 2 * e.vision + 1
        if net.policy_impl != 'tc' or not self.use_xtable or W * W > 25 or 1 + sum(self.args.naction_heads) > 8:
            return False
        if getattr(net, 'is_variant', False):          # the BPTT kernels differentiate ONE comm pass
            return False
        if getattr(e, 'obs_layout', (0, 0, 0))[1] == 0:
            return False
        npos = e.obs_positions
        used = npos + ((W * W + 4) if self.is_tj else (2 * W * W + 1))
        return (used + 15) // 16 * 16 <= 512

    def _encoder_table(self, cfg, w):
        """[positions, H] class part of x per agent position for the CURRENT weights (None when not applicable)."""
        e, net = self.env.env, self.policy_net
        if not self.use_xtable or cfg.obs_vocab == 0:
            return None
        key = net._packed_key
        if self._xtable is None:
            self._xtable = torch.empty(e.obs_positions, net.hid_size, device=e.device)
        if key != self._xtable_key:
            fn = _lib.load().ic3_tj_encoder_table if self.is_tj else _lib.load().ic3_pp_encoder_table
            _lib.check(fn(C.byref(e.cfg), C.byref(cfg), C.byref(w), self._xtable.data_ptr(), _lib.stream()))
            self._xtable_key = key
        return self._xtable

    # ------------------------------------------------------------------ buffers
    def _alloc(self, T):
        e = self.env.env
        B, N, H = e.nenvs, self.args.nagents, self.args.hid_size
        dev = e.device
        nh = len(self.args.naction_heads)
        A = sum(self.args.naction_heads)
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=dev)
        b = dict(T=T, h=z(B * N, H), c=z(B * N, H), x=z(B * N, H),
                 comm=z(B, N, dtype=torch.uint8), alive=torch.ones(B, N, dtype=torch.uint8, device=dev),
                 fresh=torch.ones(B, dtype=torch.uint8, device=dev), t_ep=z(B, dtype=torch.int32),
                 action=z(T, B, N, nh, dtype=torch.int32), logp=z(T, B, N, A), value=z(T, B * N),
                 reward=z(T, B, N), emask=z(T, B, dtype=torch.uint8), mini=z(T, B, N, dtype=torch.uint8),
                 ralive=z(T, B, N, dtype=torch.uint8), step_reward=z(B, N),
                 stat_reward=z(B, N), stat_comm=z(B, N), stat_success=z(B, dtype=torch.int32),
                 stat_episodes=z(B, dtype=torch.int32), stat_steps=z(B, dtype=torch.int32),
                 err=z(1, dtype=torch.int32), halted=z(B, dtype=torch.uint8), valid=z(T, B, dtype=torch.uint8),
                 statvec=z(4 + 2 * N, dtype=torch.float64))
        if self.obs_mode == 'dense' or (self.record_for_grad and self.is_tj and not self.grad_kernels):
            b['obs'] = torch.empty(B, N, self.env.observation_dim, dtype=torch.float32, device=dev)
        if self.record_for_grad and self.grad_kernels:
            # hand-written BPTT (csrc/bptt_tc.cu): every step's (h, c) -- the policy step writes them straight into
            # the record, rec_h[t] -> rec_h[t + 1] -- and the inputs / env state each observation was taken from
            b.update(s_fresh=z(T, B, dtype=torch.uint8), s_comm=z(T, B, N, dtype=torch.uint8),
                     s_alive=z(T, B, N, dtype=torch.uint8), s_tep=z(T, B, dtype=torch.int32),
                     rec_h=torch.empty(T + 1, B * N, H, device=dev), rec_c=torch.empty(T + 1, B * N, H, device=dev))
            if self.is_tj:
                b.update(s_tjloc=z(T, B, N, 2, dtype=torch.int32), s_tjalive=z(T, B, N, dtype=torch.uint8),
                         s_tjlast=z(T, B, N, dtype=torch.uint8), s_tjroute=z(T, B, N, dtype=torch.int32))
            else:
                b['s_loc'] = z(T, B, e.npredator + 1, 2, dtype=torch.int32)    # predators + the prey
        elif self.record_for_grad:
            # inputs of every policy step + (h, c) checkpoints at the window starts
            W = self.grad_window
            nw = (T + W - 1) // W
            b.update(s_fresh=z(T, B, dtype=torch.uint8), s_comm=z(T, B, N, dtype=torch.uint8),
                     s_alive=z(T, B, N, dtype=torch.uint8), s_tep=z(T, B, dtype=torch.int32),
                     ck_h=z(nw, B * N, H), ck_c=z(nw, B * N, H))
            if self.is_tj:
                b['s_obs'] = z(T, B, N, self.env.observation_dim)
            else:
                b['s_loc'] = z(T, B, e.npredator + 1, 2, dtype=torch.int32)    # predators + the prey
        self._buf = b
        self._graph = None
        return b

    # ------------------------------------------------------------------ rollout
    def _dense_chunks(self, cfg):
        """[(env cfg, env state, policy cfg, obs ptr, x ptr)] per chunk of env slots; chunk bytes <= obs_chunk_mb."""
        e, b = self.env.env, self._buf
        B, N, O, H = e.nenvs, self.args.nagents, self.env.observation_dim, self.args.hid_size
        key = (B, b['obs'].data_ptr(), b['x'].data_ptr(), cfg.obs_vocab, cfg.seed, cfg.env_id0)
        if getattr(self, '_chunks_key', None) == key:
            return self._chunks
        # default: ONE chunk.  Measured on B200 (PP hard, 1.19 GB of observations per step): 18 chunks of 64 MB run the
        # step in 0.70 ms (0.60 ms as a CUDA graph) against 0.55 ms (0.53 ms) for the whole batch -- the tails of 36
        # small kernels cost more than the L2 hits save.  Batches that fit in L2 anyway (traffic junction) get the
        # benefit without chunking: the gather kernel keeps them in L2 by itself (IC3_OBS_L2_KEEP_BYTES).
        mb = float(getattr(self.args, 'obs_chunk_mb', 0) or 0)
        per_env = N * O * 4
        nchunk = max(1, -(-B * per_env // int(mb * (1 << 20)))) if mb > 0 else 1
        step = -(-B // nchunk)
        out = []
        for k0 in range(0, B, step):
            k1 = min(B, k0 + step)
            ecfg, est = e.chunk_view(k0, k1)
            ccfg = _lib.PolicyCfg.from_buffer_copy(cfg)
            ccfg.B, ccfg.env_id0 = k1 - k0, cfg.env_id0 + k0
            out.append((ecfg, est, ccfg, b['obs'].data_ptr() + k0 * per_env, b['x'].data_ptr() + k0 * N * H * 4))
        self._chunks, self._chunks_key = out, key
        return out

    def _fused_x(self):
        """Index-form observations on the tensor-core policy path: the encoder runs inside the policy step."""
        dense = self.obs_mode == 'dense' or (self.record_for_grad and self.is_tj and not self.grad_kernels)
        W = 2 * self.env.env.vision + 1
        return (not dense) and self.policy_net.policy_impl == 'tc' and W * W <= 25

    def _enqueue(self, T, quota=0):
        """Enqueue T lock-step iterations on the current stream (no host sync).  quota > 0: reference batch
        boundary -- a slot halts at the first episode end with >= quota steps (ic3_rollout_io.batch_size);
        quota = 0: episodes still open at iteration T-1 are cut there."""
        b, e, net, args = self._buf, self.env.env, self.policy_net, self.args
        lib = _lib.load()
        B, N = e.nenvs, args.nagents
        nh = len(args.naction_heads)
        cfg = net.policy_cfg(B)
        cfg.seed, cfg.env_id0 = e.cfg.seed, e.cfg.env_id0
        w = net.packed()
        hard = int(bool(args.hard_attn) and bool(args.commnet))
        s = _lib.stream()
        ws, _ = net.workspace(B)          # tensor-core path scratch (None for the fp32 SIMT kernel)
        rec = self.record_for_grad
        gk = rec and self.grad_kernels
        dense = self.obs_mode == 'dense' or (rec and self.is_tj and not gk)
        # tensor-core path: the index encoder is fused into the policy step (x never leaves the operand image)
        fused_x = self._fused_x()
        src = {}
        if fused_x:
            src = dict(tj_env=C.addressof(e.cfg), tj_state=C.addressof(e.state)) if self.is_tj else \
                dict(pp_env=C.addressof(e.cfg), pp_state=C.addressof(e.state))
            src['x_table'] = _lib.ptr(self._encoder_table(cfg, w))
        snap = {}
        if rec:
            snap = dict(snap_T=T, snap_fresh=b['s_fresh'].data_ptr(), snap_comm=b['s_comm'].data_ptr(),
                        snap_alive=b['s_alive'].data_ptr(), snap_tep=b['s_tep'].data_ptr())
            if not self.is_tj:
                snap['snap_pp_loc'] = b['s_loc'].data_ptr()
            elif gk:
                snap.update(snap_tj_loc=b['s_tjloc'].data_ptr(), snap_tj_alive=b['s_tjalive'].data_ptr(),
                            snap_tj_last_act=b['s_tjlast'].data_ptr(), snap_tj_route_id=b['s_tjroute'].data_ptr())
        for t in range(T):
            if rec:
                if t == 0:          # inputs of the first step; the env step kernels record those of every later step
                    b['s_fresh'][0].copy_(b['fresh'])
                    b['s_comm'][0].copy_(b['comm'])
                    b['s_alive'][0].copy_(b['alive'])
                    b['s_tep'][0].copy_(b['t_ep'])
                    if not self.is_tj:
                        b['s_loc'][0].copy_(e.loc)
                    elif gk:
                        b['s_tjloc'][0].copy_(e.car_loc)
                        b['s_tjalive'][0].copy_(e.alive_mask)
                        b['s_tjlast'][0].copy_(e.car_last_act)
                        b['s_tjroute'][0].copy_(e.route_id)
                if not gk and t % self.grad_window == 0:
                    b['ck_h'][t // self.grad_window].copy_(b['h'])
                    b['ck_c'][t // self.grad_window].copy_(b['c'])
            if dense:
                # gather + encode, optionally in chunks of env slots (args.obs_chunk_mb; default one chunk, see
                # _dense_chunks); observation batches that fit in L2 are written with plain stores and the encoder
                # reads them from L2 instead of HBM
                obs_fn = lib.ic3_tj_obs if self.is_tj else lib.ic3_pp_obs
                for ecfg, est, ccfg, o_ptr, x_ptr in self._dense_chunks(cfg):
                    _lib.check(obs_fn(C.byref(ecfg), C.byref(est), o_ptr, s))
                    _lib.check(lib.ic3_encoder_dense(C.byref(ccfg), C.byref(w), o_ptr, x_ptr, s))
                if rec and self.is_tj:
                    b['s_obs'][t].copy_(b['obs'])
            elif fused_x:
                pass
            elif self.is_tj:
                _lib.check(lib.ic3_tj_encoder_index(C.byref(e.cfg), C.byref(e.state), C.byref(cfg), C.byref(w),
                                                    b['x'].data_ptr(), s))
            else:
                _lib.check(lib.ic3_pp_encoder_index(C.byref(e.cfg), C.byref(e.state), C.byref(cfg), C.byref(w),
                                                    b['x'].data_ptr(), s))
            hin, cin = (b['rec_h'][t], b['rec_c'][t]) if gk else (b['h'], b['c'])
            hout, cout = (b['rec_h'][t + 1], b['rec_c'][t + 1]) if gk else (b['h'], b['c'])
            io = _lib.PolicyIO(x=None if fused_x else b['x'].data_ptr(), h=hin.data_ptr(), c=cin.data_ptr(),
                               comm_action=b['comm'].data_ptr() if hard else None, alive=b['alive'].data_ptr(),
                               fresh=b['fresh'].data_ptr(), tick=e.tick.data_ptr(), draws=None,
                               h_out=hout.data_ptr(), c_out=cout.data_ptr(), value=b['value'][t].data_ptr(),
                               logp=b['logp'][t].data_ptr(), action=b['action'][t].data_ptr(),
                               workspace=_lib.ptr(ws), err=b['err'].data_ptr(), **src)
            _lib.check(lib.ic3_policy_step(C.byref(cfg), C.byref(w), C.byref(io), s))
            r = _lib.RolloutIO(t=t, max_steps=args.max_steps, nheads=nh, hard_attn=hard,
                               comm_action_one=int(bool(args.comm_action_one)),
                               last=int(t == T - 1 and quota <= 0), batch_size=int(quota),
                               halted=b['halted'].data_ptr(), rec_valid=b['valid'].data_ptr(), **snap,
                               action=b['action'][t].data_ptr(), t_ep=b['t_ep'].data_ptr(),
                               fresh=b['fresh'].data_ptr(), comm_next=b['comm'].data_ptr(),
                               alive_next=b['alive'].data_ptr(), rec_reward=b['reward'].data_ptr(),
                               rec_episode_mask=b['emask'].data_ptr(), rec_mini_mask=b['mini'].data_ptr(),
                               rec_alive=b['ralive'].data_ptr(), stat_reward=b['stat_reward'].data_ptr(),
                               stat_comm=b['stat_comm'].data_ptr(), stat_success=b['stat_success'].data_ptr(),
                               stat_episodes=b['stat_episodes'].data_ptr(), stat_steps=b['stat_steps'].data_ptr())
            if self.is_tj:
                _lib.check(lib.ic3_tj_step(C.byref(e.cfg), C.byref(e.state), b['action'][t].data_ptr(), nh, None,
                                           b['step_reward'].data_ptr(), None, b['err'].data_ptr(), C.byref(r), s))
            else:
                _lib.check(lib.ic3_pp_step(C.byref(e.cfg), C.byref(e.state), b['action'][t].data_ptr(), nh,
                                           b['step_reward'].data_ptr(), None, b['err'].data_ptr(), C.byref(r), s))

    def _episode_boundary(self, epoch):
        e, b = self.env.env, self._buf
        if self.is_tj:
            e.reset(epoch, want_obs=False)
        else:
            e.reset(want_obs=False)
        for k in ('stat_reward', 'stat_comm', 'stat_success', 'stat_episodes', 'stat_steps', 't_ep', 'halted'):
            b[k].zero_()
        b['fresh'].fill_(1)

    def rollout(self, T, epoch=0, quota=0):
        """T lock-step iterations from fresh episodes in every slot (``quota``: see _enqueue).  Returns a
        RolloutBatch of stacked [T, B, ...] device tensors (views of the trainer's record buffers)."""
        e = self.env.env
        if self._buf is None or self._buf['T'] != T:
            self._alloc(T)
        b = self._buf
        self._episode_boundary(epoch)             # trainer.py:28-32, 45-51
        b['err'].zero_()
        w = self.policy_net.packed()              # (re)pack weights outside any graph capture
        if self._fused_x():
            self._encoder_table(self.policy_net.policy_cfg(e.nenvs), w)  # ... and the encoder table with them
        if self.use_graph:
            # kernel arguments passed BY VALUE are frozen into a captured graph: everything of that kind that can
            # change between rollouts is part of the key (the TJ curriculum moves cfg.spawn_thr, traffic_junction_env.py:
            # 196-200,620-626; a re-seeded env changes cfg.seed) and a stale graph is re-captured
            key = (T, int(quota), int(getattr(e.cfg, 'spawn_thr', 0)), int(e.cfg.seed), int(e.cfg.env_id0))
            if self._graph is None or self._graph_key != key:
                # warm-up pass (lazy function attributes, allocator) on a snapshot of the env state, rewound afterwards:
                # the captured pass then starts from exactly the state an eager rollout would start from (same RNG ticks)
                snap = e.snapshot()
                keys = ('fresh', 'comm', 'alive', 't_ep', 'h', 'c', 'halted', 'stat_reward', 'stat_comm', 'stat_success',
                        'stat_episodes', 'stat_steps')
                saved = {k: b[k].clone() for k in keys}
                self._enqueue(T, quota)
                torch.cuda.synchronize()
                e.restore(snap)                   # env state, RNG ticks ...
                for k, v in saved.items():        # ... and the trainer-side episode state, as the boundary above left them
                    b[k].copy_(v)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._enqueue(T, quota)
                self._graph, self._graph_key = g, key
                g.replay()
            else:
                self._graph.replay()
        else:
            self._enqueue(T, quota)
        return RolloutBatch(action=b['action'], logp=b['logp'], value=b['value'].view(T, e.nenvs, -1),
                            reward=b['reward'], episode_mask=b['emask'], episode_mini_mask=b['mini'],
                            alive_mask=b['ralive'], valid=b['valid'])

    def stat_vector(self):
        """Device float64 vector [num_episodes, num_steps, success, err flags, reward[N], comm_action[N]] of this
        GPU's slots (one kernel, csrc/returns.cu ic3_stat_reduce); no host synchronisation."""
        b, e = self._buf, self.env.env
        hard = bool(self.args.hard_attn) and bool(self.args.commnet)
        _lib.check(_lib.load().ic3_stat_reduce(e.nenvs, self.args.nagents, b['stat_episodes'].data_ptr(),
                                               b['stat_steps'].data_ptr(), b['stat_success'].data_ptr(),
                                               b['err'].data_ptr(), b['stat_reward'].data_ptr(),
                                               b['stat_comm'].data_ptr() if hard else None,
                                               b['statvec'].data_ptr(), _lib.stream()))
        return b['statvec']

    def stat_from_vector(self, v):
        """Host-side stat dict with the reference's keys (trainer.py:73-75,86-88,109-110,124-125,235) from a
        stat_vector() (of this GPU, or summed over ranks) that has been copied to the host."""
        args, N = self.args, self.args.nagents
        flags = int(v[3])
        if flags:
            raise RuntimeError("device-side error flag %#x during rollout" % flags)
        stat = dict()
        stat['num_episodes'] = int(round(float(v[0])))
        stat['num_steps'] = int(round(float(v[1])))
        stat['steps_taken'] = stat['num_steps']
        nf = int(getattr(args, 'nfriendly', N))                 # trainer.py:73-75,86-88: friendly / enemy split
        enemy = bool(getattr(args, 'enemy_comm', False))
        stat['reward'] = v[4:4 + nf].copy()
        if enemy:
            stat['enemy_reward'] = v[4 + nf:4 + N].copy()
        if args.hard_attn and args.commnet:
            stat['comm_action'] = v[4 + N:4 + N + nf].copy()
            if enemy:
                stat['enemy_comm'] = v[4 + N + nf:4 + 2 * N].copy()
        if not (not self.is_tj and args.mode == 'competitive'):
            stat['success'] = int(round(float(v[2])))
        if self.is_tj:
            # every episode of the batch reports the same env.stat['add_rate'] (traffic_junction_env.py:249-250),
            # merged by + over episodes and workers (trainer.py:124-125, utils.py:15-29)
            stat['add_rate'] = self.env.env.add_rate * stat['num_episodes']
        return stat

    def collect_stat(self):
        """Stat dict of the last rollout, summed over the env slots of this GPU (ONE device->host copy)."""
        return self.stat_from_vector(self.stat_vector().cpu().numpy())

    # ------------------------------------------------------------------ reference surface
    def get_episode(self, epoch):
        """Exactly one episode per env slot (trainer.py:26-126): max_steps lock-step iterations, a slot whose
        episode ends early halts (``valid`` = 0 afterwards)."""
        batch = self.rollout(self.args.max_steps, epoch, quota=1)
        return batch, self.collect_stat()

    def episodes_end_early(self):
        """Can an episode end before max_steps?  predator_prey 'mixed' mode only (predator_prey_env.py:273-274);
        traffic_junction never sets episode_over (traffic_junction_env.py:219,252)."""
        return (not self.is_tj) and getattr(self.args, 'mode', 'mixed') == 'mixed'

    def batch_plan(self):
        """(lock-step iterations, quota) of one run_batch."""
        bs, ms = int(self.args.batch_size), int(self.args.max_steps)
        full = int(math.ceil(bs / float(ms))) * ms
        if getattr(self.args, 'batch_boundary', 'reference') == 'cut':
            return full, 0
        return (bs + ms - 1 if self.episodes_end_early() else full), bs

    def steps_per_batch(self):
        return self.batch_plan()[0]

    def run_batch(self, epoch):
        T, quota = self.batch_plan()
        batch = self.rollout(T, epoch, quota=quota)
        self.stats = self.collect_stat()
        return batch, self.stats

    # ------------------------------------------------------------------ gradient (trainer.py:128-225)
    def _pp_sparse_obs(self, loc):
        """Non-zeros of the PP observation (predator_prey_env.py:188-210) as (index, value) pairs
        [R, 3*W*W] from a state snapshot loc [B, N+1, 2]."""
        e = self.env.env
        D, v, N = e.dim, e.vision, e.npredator
        NA = e.nagent_rows                                                   # + the prey's own row with enemy_comm
        W, V = 2 * v + 1, e.vocab_size
        loc = loc.long()
        pr, pc = loc[:, :N, 0], loc[:, :N, 1]
        ar = torch.arange(W, device=loc.device)
        dy, dx = ar.repeat_interleave(W), ar.repeat(W)                       # window cell w = dy*W + dx
        rr = loc[:, :NA, 0].unsqueeze(-1) - v + dy                           # [B, NA, W*W]
        cc = loc[:, :NA, 1].unsqueeze(-1) - v + dx
        inside = (rr >= 0) & (rr < D) & (cc >= 0) & (cc < D)
        base = torch.arange(W * W, device=loc.device) * V
        cls = torch.where(inside, rr * D + cc, torch.full_like(rr, D * D + 1)) + base
        npred = ((rr.unsqueeze(-1) == pr[:, None, None, :]) & (cc.unsqueeze(-1) == pc[:, None, None, :])).sum(-1)
        nprey = (rr == loc[:, N:, 0].unsqueeze(-1)) & (cc == loc[:, N:, 1].unsqueeze(-1))
        idx = torch.cat([cls, (base + V - 2).expand_as(cls), (base + V - 1).expand_as(cls)], -1)
        val = torch.cat([torch.ones_like(cls), nprey.long() * inside, npred * inside], -1).float()
        return idx.reshape(-1, 3 * W * W), val.reshape(-1, 3 * W * W)

    def _forward_window(self, t0, t1, h, c, adv, ret):
        """Differentiable re-run of steps [t0, t1) for all slots; returns (loss, h, c, stats)."""
        b, net, args = self._buf, self.policy_net, self.args
        B, N, H = self.env.env.nenvs, args.nagents, args.hid_size
        hard = bool(args.hard_attn) and bool(args.commnet)
        w = net._kernel_weights()
        w_e, b_e = w['enc_w'], w['enc_b']
        w_eT = None if self.is_tj else w_e.t().contiguous()
        loss = torch.zeros((), device=h.device)
        st = dict(action_loss=torch.zeros((), device=h.device), value_loss=torch.zeros((), device=h.device),
                  entropy=torch.zeros((), device=h.device))
        for t in range(t0, t1):
            keep = (1 - b['s_fresh'][t].float()).repeat_interleave(N).unsqueeze(1)        # trainer.py:50-51
            h, c = h * keep, c * keep
            if self.is_tj:
                x = F.linear(b['s_obs'][t].reshape(B * N, -1), w_e, b_e)                  # comm.py:119
            else:
                idx, val = self._pp_sparse_obs(b['s_loc'][t])
                x = F.embedding_bag(idx, w_eT, per_sample_weights=val, mode='sum') + b_e
            fresh = b['s_fresh'][t].bool().unsqueeze(1)
            alive = torch.where(fresh, torch.ones_like(b['s_alive'][t]), b['s_alive'][t]).float()   # comm.py:99-112
            n_alive = alive.sum(1, keepdim=True)
            g = alive
            if hard:
                g = g * torch.where(fresh, torch.zeros_like(b['s_comm'][t]), b['s_comm'][t]).float()  # :171-175
            h, c, value, logps = policy_forward_torch(net, x, h, c, g, n_alive)
            value = value.view(B, N)
            alive_post = b['ralive'][t].float()
            act = b['action'][t].long()
            lp_taken = torch.zeros(B, N, device=h.device)
            ent = torch.zeros((), device=h.device)
            vmask = b['valid'][t].float().view(B, 1, 1)            # 0 for slots that already completed their batch
            for k, lp in enumerate(logps):
                lp = lp.view(B, N, -1)                                                     # comm.py:239
                lp_taken = lp_taken + lp.gather(-1, act[..., k:k + 1]).squeeze(-1)         # utils.py:42-46
                ent = ent - (lp * lp.exp() * vmask).sum()
            a_loss = (-adv[t] * lp_taken * alive_post).sum()                               # trainer.py:198-201
            v_loss = ((value - ret[t]).pow(2) * alive_post).sum()                          # :205-208
            step_loss = a_loss + args.value_coeff * v_loss
            if args.entr > 0:
                step_loss = step_loss - args.entr * ent                                    # :211-220
            loss = loss + step_loss
            st['action_loss'] += a_loss.detach(); st['value_loss'] += v_loss.detach(); st['entropy'] += ent.detach()
            det = (((b['s_tep'][t] + 1) % args.detach_gap) == 0).repeat_interleave(N).unsqueeze(1)   # trainer.py:56-60
            if bool(args.detach_gap <= self.args.max_steps):
                h = torch.where(det, h.detach(), h)
                c = torch.where(det, c.detach(), c)
        return loss, h, c, st

    LOSS_KEYS = ('action_loss', 'value_loss', 'entropy')

    def compute_grad(self, batch):
        """REINFORCE + value + entropy loss summed over every slot and step of the batch, gradients
        accumulated into ``p.grad`` (not yet divided by num_steps: train_batch does that,
        trainer.py:251-253).  Needs ``args.record_for_grad`` during the rollout.  Returns the reference's stat
        dict (trainer.py:222-225)."""
        v = self.compute_grad_device(batch).cpu().numpy()
        return {k: float(v[i]) for i, k in enumerate(self.LOSS_KEYS)}

    def compute_grad_device(self, batch):
        """compute_grad without a host synchronisation: the three loss sums come back as a float64 DEVICE vector
        (LOSS_KEYS order) so the data-parallel trainer can reduce them together with the batch statistics."""
        if not self.record_for_grad:
            raise RuntimeError("set args.record_for_grad = True before the rollout to use compute_grad")
        b, args = self._buf, self.args
        e = self.env.env
        T, B, N = b['T'], e.nenvs, args.nagents
        ret = torch.empty(T, B, N, device=e.device)
        _lib.check(_lib.load().ic3_returns_scan(T, B, N, float(args.gamma), float(args.mean_ratio),
                                                b['reward'].data_ptr(), b['emask'].data_ptr(), b['mini'].data_ptr(),
                                                ret.data_ptr(), _lib.stream()))
        adv = ret - b['value'].view(T, B, N)                                               # trainer.py:176-177
        if args.normalize_rewards:                                   # :179-180, per slot, over its REAL steps only
            v = b['valid'].float().unsqueeze(-1)                     # [T, B, 1]
            cnt = v.sum(0, keepdim=True) * N
            mean = (adv * v).sum((0, 2), keepdim=True) / cnt
            var = (((adv - mean) * v) ** 2).sum((0, 2), keepdim=True) / (cnt - 1)      # torch.std: unbiased
            adv = (adv - mean) / var.sqrt()
        if self.grad_kernels:
            return self._compute_grad_kernels(adv, ret)
        W = self.grad_window
        nw = (T + W - 1) // W
        dh = dc = None
        if self.grad_impl == 'manual':
            tot = self._compute_grad_manual(adv, ret, W, nw)
            return torch.tensor([tot[k] for k in self.LOSS_KEYS], dtype=torch.float64, device=e.device)
        tot = torch.zeros(3, dtype=torch.float64, device=e.device)
        for k in reversed(range(nw)):
            t0, t1 = k * W, min(T, (k + 1) * W)
            h0 = b['ck_h'][k].clone().requires_grad_(True)
            c0 = b['ck_c'][k].clone().requires_grad_(True)
            loss, h1, c1, st = self._forward_window(t0, t1, h0, c0, adv, ret)
            if dh is not None:                     # gradient arriving from the later window
                loss = loss + (h1 * dh).sum() + (c1 * dc).sum()
            loss.backward()
            # variants without a cell state / without a carried hidden state leave these gradients undefined: zero
            dh = h0.grad.detach() if h0.grad is not None else torch.zeros_like(h0)
            dc = c0.grad.detach() if c0.grad is not None else torch.zeros_like(c0)
            tot += torch.stack([st[key] for key in self.LOSS_KEYS]).double()
        return tot

    def _compute_grad_kernels(self, adv, ret):
        """Hand-written BPTT (csrc/bptt_tc.cu): one ic3_bptt_step per lock-step iteration, last to first (one host read
        up front: max |c| of the record, the bound behind the operand scale).  Returns the device float64 vector of the
        three loss sums."""
        b, net, args, e = self._buf, self.policy_net, self.args, self.env.env
        lib = _lib.load()
        T, B, N, H = b['T'], e.nenvs, args.nagents, args.hid_size
        s = _lib.stream()
        cfg = net.policy_cfg(B)
        cfg.seed, cfg.env_id0 = e.cfg.seed, e.cfg.env_id0
        w = net.packed()
        table = self._encoder_table(cfg, w)
        if self._bptt is None or self._bptt['B'] != B:
            plan = _lib.BpttPlan(cfg=C.pointer(cfg), w=C.pointer(w),
                                 pp_env=None if self.is_tj else C.pointer(e.cfg),
                                 tj_env=C.pointer(e.cfg) if self.is_tj else None, x_table=table.data_ptr(),
                                 value_coeff=float(args.value_coeff), entr=float(args.entr), workspace=None)
            nbytes = int(lib.ic3_bptt_workspace_bytes(C.byref(plan)))
            if nbytes == 0:
                raise NotImplementedError("this configuration is outside the BPTT kernels (use grad_impl='autograd')")
            self._bptt = dict(B=B, ws=torch.empty(nbytes, dtype=torch.uint8, device=e.device),
                              dh=torch.zeros(B * N, H, device=e.device), dc=torch.zeros(B * N, H, device=e.device),
                              losses=torch.zeros(3, dtype=torch.float64, device=e.device))
        st = self._bptt
        plan = _lib.BpttPlan(cfg=C.pointer(cfg), w=C.pointer(w), pp_env=None if self.is_tj else C.pointer(e.cfg),
                             tj_env=C.pointer(e.cfg) if self.is_tj else None, x_table=table.data_ptr(),
                             value_coeff=float(args.value_coeff), entr=float(args.entr), workspace=st['ws'].data_ptr())
        hard = bool(args.hard_attn) and bool(args.commnet)
        adv = adv.contiguous()
        cut = None
        if args.detach_gap <= args.max_steps:                                  # trainer.py:56-60
            cut = (((b['s_tep'] + 1) % args.detach_gap) == 0).to(torch.uint8).contiguous()
        lo, hi = torch.aminmax(b['rec_c'][1:])                                  # bound of |c| for the operand scale
        cmax = max(abs(float(lo.item())), abs(float(hi.item())))
        st['dh'].zero_()
        st['dc'].zero_()
        _lib.check(lib.ic3_bptt_begin(C.byref(plan), cmax, s))
        value = b['value']

        def step_io(t):
            return _lib.BpttStepIO(t=t, h_prev=b['rec_h'][t].data_ptr(), c_prev=b['rec_c'][t].data_ptr(),
                                   h_new=b['rec_h'][t + 1].data_ptr(), fresh=b['s_fresh'][t].data_ptr(),
                                   comm=b['s_comm'][t].data_ptr() if hard else None, alive=b['s_alive'][t].data_ptr(),
                                   cut=cut[t].data_ptr() if cut is not None else None,
                                   pp_loc=None if self.is_tj else b['s_loc'][t].data_ptr(),
                                   tj_loc=b['s_tjloc'][t].data_ptr() if self.is_tj else None,
                                   tj_alive=b['s_tjalive'][t].data_ptr() if self.is_tj else None,
                                   tj_last_act=b['s_tjlast'][t].data_ptr() if self.is_tj else None,
                                   tj_route_id=b['s_tjroute'][t].data_ptr() if self.is_tj else None,
                                   logp=b['logp'][t].data_ptr(), action=b['action'][t].data_ptr(),
                                   value=value[t].data_ptr(), ret=ret[t].data_ptr(), adv=adv[t].data_ptr(),
                                   alive_post=b['ralive'][t].data_ptr(), valid=b['valid'][t].data_ptr(),
                                   dh=st['dh'].data_ptr(), dc=st['dc'].data_ptr(), err=b['err'].data_ptr())
        # look-ahead: the heads gradient and the operand images of step t - 1 do not depend on the recursion; they are
        # launched on the library's side stream before step t and overlap its tensor-core kernels
        nxt = step_io(T - 1) if T > 0 else None
        if nxt is not None:
            _lib.check(lib.ic3_bptt_prepare(C.byref(plan), C.byref(nxt), s))
        for t in reversed(range(T)):
            io = nxt
            if t > 0:
                nxt = step_io(t - 1)
                _lib.check(lib.ic3_bptt_prepare(C.byref(plan), C.byref(nxt), s))
            _lib.check(lib.ic3_bptt_step(C.byref(plan), C.byref(io), s))
        # parameter gradients are ADDED to the .grad buffers (flat views of FlatRMSprop)
        params, grads = self._param_structs()
        _lib.check(lib.ic3_bptt_finish(C.byref(plan), C.byref(params), C.byref(grads), st['losses'].data_ptr(), s))
        return st['losses']

    def _param_structs(self):
        """ic3_policy_params of the parameters and of their gradient buffers (reference layouts), by kernel role."""
        net = self.policy_net
        w = net._kernel_weights()
        scratch = self.__dict__.setdefault('_grad_scratch', {})

        def grad_ptr(p):
            if isinstance(p, torch.nn.Parameter):
                if p.grad is None:
                    p.grad = torch.zeros_like(p)
                return p.grad.data_ptr()
            key = p.data_ptr()                       # frozen buffer (models.py: zero comm projection): discard its gradient
            if key not in scratch:
                scratch[key] = torch.zeros_like(p)
            return scratch[key].data_ptr()

        def mk(get):
            arr = lambda lst: (C.c_void_p * _lib.MAX_HEADS)(*([get(t) for t in lst] + [None] * (_lib.MAX_HEADS - len(lst))))
            return _lib.PolicyParams(encoder_w=get(w['enc_w']), encoder_b=get(w['enc_b']), c_w=get(w['c_w'][0]),
                                     c_b=get(w['c_b'][0]), w_ih=get(w['w_ih']), w_hh=get(w['w_hh']), b_ih=get(w['b_ih']),
                                     b_hh=get(w['b_hh']), value_w=get(w['value_w']), value_b=get(w['value_b']),
                                     head_w=arr(w['head_w']), head_b=arr(w['head_b']))
        return mk(lambda p: p.data_ptr()), mk(grad_ptr)

    def _compute_grad_manual(self, adv, ret, W, nw):
        """``args.grad_impl == 'manual'``: the same gradient from the explicit backward formulas of bptt.py (no autograd
        graph; validated in float64 against the oracle by tests/test_bptt_manual.py).  Opt-in until it has been
        measured on the GPU."""
        from . import bptt
        b, net, args = self._buf, self.policy_net, self.args
        if getattr(net, 'is_variant', False) or type(net).__name__ != 'CommNetMLP':
            raise NotImplementedError("grad_impl='manual' covers the recurrent LSTM CommNet / IC3Net with one comm pass")
        B, N = self.env.env.nenvs, args.nagents
        T = b['T']
        P, G = {}, {}
        for name, p in net.named_parameters():
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            P[name], G[name] = p.detach(), p.grad
        spec = bptt.Spec(N, args.hid_size, len(args.naction_heads), bool(args.hard_attn) and bool(args.commnet),
                         getattr(args, 'comm_mode', 'avg') == 'avg', bool(args.comm_mask_zero), args.value_coeff,
                         args.entr, args.detach_gap, args.max_steps)
        if self.is_tj:
            obs_fn = lambda t: b['s_obs'][t].reshape(B * N, -1)
        else:
            obs_fn = lambda t: self._pp_sparse_obs(b['s_loc'][t])
        rec = dict(fresh=b['s_fresh'], comm=b['s_comm'], alive=b['s_alive'], t_ep=b['s_tep'], action=b['action'],
                   alive_post=b['ralive'], obs=obs_fn, valid=b['valid'])
        tot = dict(action_loss=0.0, value_loss=0.0, entropy=0.0)
        dh = dc = None
        for k in reversed(range(nw)):
            t0, t1 = k * W, min(T, (k + 1) * W)
            dh, dc, st = bptt.window_backward(P, G, spec, rec, t0, t1, b['ck_h'][k], b['ck_c'][k], adv, ret, dh, dc)
            for key in tot:
                tot[key] += st[key]
        return tot

    # only used when there is a single process (trainer.py:245-256)
    def train_batch(self, epoch):
        batch, stat = self.run_batch(epoch)
        self.optimizer.zero_grad(set_to_none=False)
        s = self.compute_grad(batch)
        merge_stat(s, stat)
        self.optimizer.step(grad_div=stat['num_steps'])      # grad /= num_steps, then the update (trainer.py:251-254)
        return stat

    def state_dict(self):
        return self.optimizer.state_dict()

    def load_state_dict(self, state):
        self.optimizer.load_state_dict(state)
