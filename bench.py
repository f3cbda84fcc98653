#!/usr/bin/env python
"""Benchmark of the IC3Net rollout hot path on B200 (BASELINE.json metric:
agent-env-steps/sec at 1/2/4/8 B200 vs the reference CPU path).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload pp_hard_ic3net] [--impl b200|reference]
                    [--dump-outputs DIR]

A "step" is one lock-step pass of the hot path over the whole env batch of a GPU:
obs gather -> encoder -> comm/LSTM/heads/sampling -> env step (+ auto-reset), i.e.
B*N agent-env-steps.  Prints ONE JSON line (see DESIGN.md "Measurement").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "agent-env-steps/sec"

WORKLOADS = {
    # BASELINE.json configs[1]: predator_prey hard (10 agents, dim 20, vision 1, 80 steps) IC3Net, 8192 envs / GPU
    "pp_hard_ic3net": dict(env_name="predator_prey", nagents=10, dim=20, vision=1, max_steps=80, nenvs=8192,
                           ic3net=True, mode="mixed"),
    # configs[3]
    "pp_hard_commnet": dict(env_name="predator_prey", nagents=10, dim=20, vision=1, max_steps=80, nenvs=8192,
                            ic3net=False, mode="mixed"),
    # configs[2]: traffic_junction medium (README: vision 0, add_rate .05/.02)
    "tj_medium_ic3net": dict(env_name="traffic_junction", nagents=10, dim=14, vision=0, max_steps=40, nenvs=8192,
                             ic3net=True, difficulty="medium", add_rate_min=0.05, add_rate_max=0.02,
                             curr_start=0, curr_end=0),
    # configs[4]
    "tj_hard_ic3net": dict(env_name="traffic_junction", nagents=20, dim=18, vision=0, max_steps=80, nenvs=4096,
                           ic3net=True, difficulty="hard", add_rate_min=0.02, add_rate_max=0.05,
                           curr_start=250, curr_end=1250),
    # configs[0] (the reference's own CPU-runnable parity case)
    "pp_easy_ic3net": dict(env_name="predator_prey", nagents=3, dim=5, vision=0, max_steps=20, nenvs=8192,
                           ic3net=True, mode="mixed"),
}


def make_args(wl, rank=0, obs_mode="dense", nenvs=None):
    d = dict(hid_size=128, recurrent=True, rnn_type="LSTM", commnet=True, hard_attn=False, comm_action_one=False,
             comm_mode="avg", comm_passes=1, comm_mask_zero=False, comm_init="uniform", share_weights=False,
             continuous=False, batch_size=500, lrate=1e-3, nenemies=1, no_stay=False, moving_prey=False,
             enemy_comm=False, mode="mixed", vocab_type="bool", add_rate_min=0.05, add_rate_max=0.2, curr_start=0,
             curr_end=0, difficulty="easy", seed=1, mean_ratio=1.0, obs_mode=obs_mode, use_graph=False)
    d.update(WORKLOADS[wl])
    if nenvs:
        d["nenvs"] = nenvs
    a = argparse.Namespace(**d)
    if a.ic3net:                       # main.py:115-123
        a.hard_attn, a.mean_ratio = True, 0
        if a.env_name == "traffic_junction":
            a.comm_action_one = True
    a.nfriendly = a.nagents
    a.env_id0 = rank * a.nenvs
    return a


def heads_of(a):
    na = 5 if a.env_name == "predator_prey" else 2
    return [na, 2] if a.hard_attn else [na]


# ------------------------------------------------------------------------------
# CPU arm (oracle port of the reference, one env per process)
# ------------------------------------------------------------------------------
def cpu_cfg(wl):
    a = make_args(wl)
    args = {k: v for k, v in vars(a).items() if isinstance(v, (int, float, str, bool))}
    cfg = dict(args=args, heads=heads_of(a))
    if a.env_name == "traffic_junction":
        cfg["tables"] = os.path.join(ROOT, "tests", "golden", "tj_tables_%s_%d.npz" % (a.difficulty, a.dim))
    return cfg


def run_cpu(wl, nprocs, budget_s, nsamples=1):
    """Run in a fresh interpreter so no CUDA context is ever forked/shared."""
    out = subprocess.check_output([sys.executable, "-m", "oracle.cpu_baseline", json.dumps(cpu_cfg(wl)),
                                   str(nprocs), str(budget_s), str(nsamples)], cwd=ROOT)
    return json.loads(out.decode().strip().split("\n")[-1])


def host_cores():
    """Host threads this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period))))
    except Exception:
        pass
    return max(1, n)


REF_NPROCESSES = 16      # BASELINE.json metric: "vs reference CPU nprocesses=16" (README.md:46-48), whatever the box has


def ref_cfg(wl, batch_size=500):
    """Flags of the reference run (main.py:25-109 names) for a workload."""
    w = dict(WORKLOADS[wl])
    w.pop("nenvs")
    ic3 = w.pop("ic3net")
    d = dict(hid_size=128, recurrent=True, rnn_type="LSTM", batch_size=batch_size, seed=1, lrate=1e-3)
    d.update(w)
    d.update(dict(ic3net=True) if ic3 else dict(commnet=True))
    return d


def run_reference(wl, modes, warmup, iters, nprocesses=REF_NPROCESSES, batch_size=500):
    """The UNMODIFIED reference's MultiProcessTrainer (oracle/ref_baseline.py) in a fresh interpreter."""
    cfg = dict(args=ref_cfg(wl, batch_size), nprocesses=nprocesses, modes=modes, warmup=warmup, iters=iters)
    env = dict(os.environ, OMP_NUM_THREADS="1", MKL_NUM_THREADS="1", PYTHONWARNINGS="ignore")
    out = subprocess.check_output([sys.executable, "-m", "oracle.ref_baseline", json.dumps(cfg)], cwd=ROOT, env=env,
                                  stderr=subprocess.DEVNULL)
    return json.loads(out.decode().strip().split("\n")[-1])


def ref_rate(samples, nagents):
    steps = sum(x[0] for x in samples)
    secs = sum(x[1] for x in samples)
    return steps * nagents / secs, secs


def reference_arm(opts):
    """CPU baseline of record: the reference's own multi_processing.py path at nprocesses = 16, OMP_NUM_THREADS = 1,
    float64, on this box's host cores.  A "step" is one update call of its MultiProcessTrainer with compute_grad
    patched out, i.e. run_batch in all 16 workers (batch_size 500 env steps each) -- the like-for-like of the GPU
    arm's rollout metric; the full train_batch (rollout + backward + gradient sum + RMSprop) is timed beside it."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = host_cores()
    K, W = opts.steps, opts.warmup
    a = make_args(opts.workload)
    N = a.nagents
    r = run_reference(opts.workload, ["rollout"], W, K)
    samples = r["modes"]["rollout"]["samples"][W:]
    v, secs = ref_rate(samples, N)
    rt = run_reference(opts.workload, ["train_batch"], 1, 3)
    vt, _ = ref_rate(rt["modes"]["train_batch"]["samples"][1:], N)
    port = run_cpu(opts.workload, REF_NPROCESSES, 4.0)
    sample = ("%d processes (reference MultiProcessTrainer, unmodified, float64, OMP_NUM_THREADS=1) x %d run_batch "
              "calls of batch_size 500 env steps each" % (REF_NPROCESSES, K))
    line = dict(metric=METRIC, value=v, unit="agent-env-steps/s", n_gpus=opts.gpus, steps=K, warmup=W,
                ms_per_step=1e3 * secs / K, higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f64", data="synthetic", impl="reference",
                config=dict(workload=opts.workload, nprocesses=REF_NPROCESSES, envs_per_process=1, nagents=N,
                            max_steps=a.max_steps, batch_size=500, host_cores=cores),
                cpu_baseline=dict(value=v, unit="agent-env-steps/s", cores=min(cores, REF_NPROCESSES),
                                  nprocesses=REF_NPROCESSES, kind="reference", sample=sample),
                train_batch=dict(value=vt, unit="agent-env-steps/s",
                                 sample="3 full train_batch calls after 1 warm-up (rollout + compute_grad + gradient "
                                        "sum over the 16 workers + RMSprop)"),
                port=dict(value=port["value"], unit="agent-env-steps/s", nprocesses=REF_NPROCESSES, kind="port",
                          sample="oracle restatement of get_episode, %d processes x 4 s" % REF_NPROCESSES),
                e2e=dict(value=v, unit="agent-env-steps/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        try:
            for ln in self.proc.stdout:
                self.rows.append([x.strip() for x in ln.decode().strip().split(",")] + [time.time()])
        except Exception:
            pass

    def __enter__(self):
        try:    # one streaming nvidia-smi (a sample every 50 ms) for the duration of the timed region
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL)
            self.th.start()
            time.sleep(0.3)
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *e):
        if self.proc is not None:
            self.proc.terminate()          # exact PID we started
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.th.join(timeout=5)

    def summary(self, window=None):
        """Median SM clock and throttle reasons over the samples that arrived inside `window`
        (wall-clock start/end of the timed region; a sample lags the GPU state by <= 50 ms)."""
        rows = self.rows
        if window is not None:
            inside = [r for r in rows if window[0] <= r[-1] <= window[1] + 0.06]
            rows = inside or rows
        sm = sorted(int(float(r[0])) for r in rows if r and str(r[0]).replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in rows if len(r) > 1 and str(r[1]).replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in rows)]
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons,
                    samples=len(rows))


# ------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------
def gpu_arm(opts):
    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    from ic3net_b200 import _lib, data
    from ic3net_b200.action_utils import parse_action_args, select_action
    from ic3net_b200.comm import CommNetMLP
    from ic3net_b200.multi_gpu import MultiGPUTrainer
    from ic3net_b200.trainer import Trainer

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # ONE JSON line on stdout is the contract: libraries that write to file descriptor 1 on their own (NCCL's version
    # banner) are sent to stderr for the whole run; the result line goes to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    # Host-side work is a few tiny tensor ops per step; letting torch fan them out over every visible
    # core (128 here, with a 16-core cgroup quota) only earns CPU throttling stalls.  The reference's
    # README asks for OMP_NUM_THREADS=1 as well (README.md:48); torchrun sets the same default.
    torch.set_num_threads(1)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # keep NCCL's version banner off stdout: ONE JSON line is the contract
        dist.init_process_group("nccl", device_id=dev)
    K, W = opts.steps, max(3, opts.warmup)

    def build(obs_mode, nenvs=None, **extra):
        a = make_args(opts.workload, rank, obs_mode, nenvs)
        a.policy_impl = opts.policy_impl
        a.obs_chunk_mb = opts.obs_chunk_mb
        a.fuse_heads = bool(int(os.environ.get("IC3_FUSE_HEADS", "0")))      # experiment: heads finished in the env step
        for k, v in extra.items():
            setattr(a, k, v)
        env = data.init(a.env_name, a)
        a.num_inputs = env.observation_dim
        a.num_actions = [env.num_actions] + ([2] if a.hard_attn else [])
        a.dim_actions = len(a.num_actions)
        parse_action_args(a)
        torch.manual_seed(0)            # random-init weights of the reference architecture, identical on every rank
        net = CommNetMLP(a, a.num_inputs)
        return a, env, net, Trainer(a, net, env)

    a, env, net, tr = build(opts.obs_mode)
    mgt = MultiGPUTrainer(a, lambda: tr)                      # broadcasts rank 0's parameters (no-op at N = 1)
    B, N, H, O = a.nenvs, a.nagents, a.hid_size, a.num_inputs
    chunk = a.max_steps                                      # record buffers hold one episode horizon
    use_graph = not opts.no_graph

    class Runner(object):
        """K lock-step iterations of a trainer, eagerly or as CUDA-graph replays (one graph per distinct length)."""

        def __init__(self, trn):
            self.trn, self.graphs, self.replayed = trn, {}, 0
            self.last_t = None                               # record index of the last enqueued iteration

        def _capture(self, n):
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            l0 = _lib.launch_count()
            with torch.cuda.graph(g):
                self.trn._enqueue(n)
            self.graphs[n] = (g, _lib.launch_count() - l0)

        def warm(self, steps):
            self.trn._alloc(chunk)
            e = self.trn.env.env
            e.reset(want_obs=False) if self.trn.args.env_name == "predator_prey" else e.reset(0, want_obs=False)
            self.trn.policy_net.packed()
            self.trn._enqueue(max(3, steps))                 # eager warm-up (lazy attributes, allocator, table)
            if use_graph:
                done = 0
                while done < K:
                    n = min(chunk, K - done)
                    if n not in self.graphs:
                        self._capture(n)
                    done += n
                self.enqueue(K)                              # one replayed pass before anything is timed
            torch.cuda.synchronize()

        def enqueue(self, steps):
            done = 0
            while done < steps:                              # episode-horizon chunks reuse the record buffers
                n = min(chunk, steps - done)
                if use_graph and n in self.graphs:
                    self.graphs[n][0].replay()               # one launch per chunk
                    self.replayed += self.graphs[n][1]
                else:
                    self.trn._enqueue(n)
                done += n
                self.last_t = n - 1

        def launches(self):
            return _lib.launch_count() + self.replayed

    def timed_region(run, steps, reduce_stats):
        """ONE timed region: K lock-step iterations + what a data-parallel update does with a rollout-only batch
        (main.py --rollout_only): the batch statistics reduced on the device and, for N > 1, the REAL collectives of
        MultiGPUTrainer -- all-reduce of the flat gradient buffer (FlatRMSprop.flat_grads, multi_processing.py:90-95)
        and of the float64 statistics vector -- then the one device->host copy of the merged statistics.
        Bracketed by barrier + synchronize on both sides; device time from CUDA events."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record()
        run.enqueue(steps)
        if reduce_stats:
            stat = mgt.reduce_device(None, with_grads=True)
        e1.record()
        torch.cuda.synchronize()
        w1 = time.time()
        if world > 1:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), (w0, w1)

    # ---- warm-up + ONE timed region of exactly K = --steps lock-step iterations (inputs resident in HBM, no host sync
    #      before the statistics copy).  A fixed step count makes the state the region leaves -- what --dump-outputs
    #      writes -- the same from run to run.  Warmed inside the clock sampler so the GPU does not idle before it, and
    #      the statistics reduction the region ends with is warmed too (first launch, first copy). ----
    run = Runner(tr)
    with ClockSampler(local) as clk:
        run.warm(W)
        mgt.reduce_device(None, with_grads=True)
        launches0 = run.launches()
        ms, window = timed_region(run, K, True)
        time.sleep(0.2)
    launches = run.launches() - launches0
    value = world * B * N * K / (ms * 1e-3)
    timing = dict(ms=ms, region="K lock-step iterations + device stat reduction"
                                + (" + all-reduce(flat_grads) + all-reduce(stat vector)" if world > 1 else "")
                                + " + 1 D2H stat copy")
    if opts.dump_outputs and rank == 0:
        dump_outputs(opts.dump_outputs, tr, run.last_t)

    # ---- full training update: MultiGPUTrainer.train_batch on every rank (rollout with the reference batch boundary
    #      + compute_grad + gradient / statistics all-reduce + RMSprop), SURVEY 8(f)-1/2 + 8(e) ----
    train = None
    skip = set(x for x in opts.skip.split(",") if x)
    if opts.quick:
        skip |= {"train", "e2e", "index", "cpu"}
    if "train" not in skip and opts.train_updates > 0:
        train = train_leg(opts, build, MultiGPUTrainer, world, dev, dist, torch)

    # ---- e2e: the public, reference-shaped API with host-side actions / rewards, on EVERY rank ----
    e2e = None
    if "e2e" not in skip:
        if world > 1:
            dist.barrier()
        # the framework's public API hands observations over as HANDLES on the env state (args.obs_api = 'handle',
        # ic3net_b200/lazy_obs.py: env.step returns a LazyObs, CommNetMLP.forward evaluates the encoder from the state,
        # bit-identical x); the dense-tensor form of the same API is timed beside it
        ah, envh, neth, trh = build(opts.obs_mode, obs_api="handle")
        mine = e2e_loop(ah, envh, neth, min(max(K, 300), 600), np, torch, select_action)
        mine["obs_api"] = "handle"
        del trh
        dense_e2e = e2e_loop(a, env, net, min(max(K, 100), 200), np, torch, select_action)
        mine["dense_obs_api"] = dict(value=dense_e2e["value"], ms_per_step=dense_e2e["ms_per_step"],
                                     note="same loop with env.step returning the dense [B,N,O] tensor (per rank)")
        try:
            mine["trainer_run_batch"] = trainer_api_leg(opts, build, world, dev, dist, torch)
        except Exception as ex:                               # e.g. no room for the pinned host copy of the batch
            mine["trainer_run_batch"] = dict(unavailable=repr(ex)[:200])
        if world > 1:
            agg = torch.tensor([mine["seconds"], float(mine["steps"])], device=dev, dtype=torch.float64)
            mx = agg.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = agg.clone()
            dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            total_steps, max_secs = float(sm[1].item()), float(mx[0].item())
            mine = dict(mine, value=total_steps * B * N / max_secs, rank0_value=mine["value"],
                        scope="all %d ranks ran the loop concurrently; value = total agent-env-steps / max wall time "
                              "over ranks" % world,
                        h2d_bytes_per_step=mine["h2d_bytes_per_step"] * world,
                        d2h_bytes_per_step=mine["d2h_bytes_per_step"] * world)
        e2e = mine

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        tc_peak = float(peaks.get("bf16_tflops", 2250.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"

        # ---- per-kernel device times (separate pass, CUDA events around every launch) ----
        kern = per_kernel_times(tr, a, env, net, min(K, 20), C, torch, _lib) if "kernels" not in skip else {}
        is_pp = a.env_name == "predator_prey"
        state_bytes = 32 if is_pp else 64
        obs_bytes = (4 * O + state_bytes) * B * N             # SURVEY 8(d): obs written once + state/action/reward
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(opts.workload, {})
        except Exception:
            pass
        roof = None
        if "obs_gather" in kern:
            ach = obs_bytes / (kern["obs_gather"] * 1e-3) / 1e9
            roof = dict(kernel="obs_gather", bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s",
                        frac=ach / hbm_peak, traffic=ncu.get("obs_gather"), peak_source=peak_src,
                        algorithmic_bytes_per_launch=obs_bytes, avg_launch_ms=kern["obs_gather"])
        kinfo = {}
        for k, v in kern.items():
            kinfo[k] = dict(avg_ms=v)
        roof_enc = None
        if "encoder_dense" in kern:
            eb = (4 * O + 4 * H) * B * N
            ach = eb / (kern["encoder_dense"] * 1e-3) / 1e9
            roof_enc = dict(kernel="encoder_dense", bound="hbm", achieved=ach, peak=hbm_peak, unit="GB/s",
                            frac=ach / hbm_peak, traffic=ncu.get("encoder_dense"), algorithmic_bytes_per_launch=eb,
                            avg_launch_ms=kern["encoder_dense"])
        roof_tc = None
        if "policy_step" in kern:
            fl = (2 * H * H + 16 * H * H) * B * N
            pb = (20 * H + 4 * (sum(a.naction_heads) + 1) + 8) * B * N
            kinfo["policy_step"].update(flops=fl, tflops=fl / (kern["policy_step"] * 1e-3) / 1e12, bytes=pb,
                                        gbs=pb / (kern["policy_step"] * 1e-3) / 1e9,
                                        math="tcgen05 kind::f16 hi/lo split, fp32 accumulate"
                                        if net.policy_impl == "tc" else "fp32 SIMT (policy v1)")
            if net.policy_impl == "tc" and "lstm_tc" in kern:
                alg = fl / (kern["lstm_tc"] * 1e-3) / 1e12
                roof_tc = dict(kernel="lstm_tc", bound="tensor", achieved=alg, issued=3 * alg, peak=tc_peak,
                               unit="TFLOP/s", frac=alg / tc_peak, frac_issued=3 * alg / tc_peak,
                               algorithmic_flops_per_launch=fl, avg_launch_ms=kern["lstm_tc"],
                               note="1x algorithmic flops (SURVEY 8(d)); the fp16 hi/lo split issues 3 MMAs per "
                                    "product; peak = measured dense bf16 cuBLAS",
                               ncu_pipe_tensor_active_pct=ncu.get("lstm_tc_pipe_tensor_pct"),
                               traffic=ncu.get("lstm_tc"))

        # ---- fused index-form rollout (no [B,N,O] tensor): the mode the trainer uses by default ----
        alt = None
        if opts.obs_mode == "dense" and world == 1 and "index" not in skip:
            a2, env2, net2, tr2 = build("index")
            run2 = Runner(tr2)
            run2.warm(W)
            ms2, _ = timed_region(run2, K, False)
            alt = dict(obs_mode="index", value=B * N * K / (ms2 * 1e-3), ms_per_step=ms2 / K,
                       note="same rollout with the encoder evaluated from the env state (bit-identical x); "
                            "this is Trainer's default obs_mode")
            del tr2, net2, env2, run2

        # ---- CPU baseline (bounded sample of the same workload on the host cores) ----
        cores = host_cores()
        cpu = None
        if world == 1 and "cpu" not in skip:
            try:
                r = run_reference(opts.workload, ["rollout"], 1, 4)
                v, secs = ref_rate(r["modes"]["rollout"]["samples"][1:], N)
                cpu = dict(value=v, unit="agent-env-steps/s", cores=min(cores, REF_NPROCESSES),
                           nprocesses=REF_NPROCESSES, kind="reference",
                           sample="reference MultiProcessTrainer (unmodified, float64, OMP_NUM_THREADS=1), %d processes "
                                  "x 4 run_batch calls of 500 env steps after 1 warm-up (%.1f s)" % (REF_NPROCESSES, secs))
            except Exception as ex:                           # staged reference missing: fall back to the port, say so
                r = run_cpu(opts.workload, REF_NPROCESSES, 8.0)
                cpu = dict(value=r["value"], unit="agent-env-steps/s", cores=min(cores, REF_NPROCESSES),
                           nprocesses=REF_NPROCESSES, kind="port",
                           sample="oracle restatement, %d processes x 8 s (reference copy unavailable: %s)"
                                  % (REF_NPROCESSES, type(ex).__name__))

        line = dict(metric=METRIC, value=value, unit="agent-env-steps/s", n_gpus=world, steps=K, warmup=W,
                    ms_per_step=ms / K, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                    data="synthetic",
                    config=dict(workload=opts.workload, envs_per_gpu=B, nagents=N, obs_dim=O, hid_size=H,
                                max_steps=a.max_steps, obs_mode=opts.obs_mode, trainer_default_obs_mode="index",
                                parallelism="dp%d" % world, cuda_graph=bool(use_graph), policy_impl=net.policy_impl,
                                l2="per-step working set %.2f GB > 126 MB L2 (inputs larger than L2)"
                                   % ((8 * O + 20 * H) * B * N / 1e9),
                                weights="random init (torch.manual_seed(0)), reference architecture"),
                    timing=timing, clocks=clk.summary(window), gpu_launches=launches, e2e=e2e, roofline=roof,
                    roofline_encoder_dense=roof_enc, roofline_tensor=roof_tc, kernels=kinfo)
        if train:
            line["train_batch"] = train
        if alt:
            line["fused_index_rollout"] = alt
        if cpu:
            line["cpu_baseline"] = cpu
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


HIDDEN_SAMPLE_SLOTS = 1024       # env slots of the hidden state written by --dump-outputs (all of them: 84 MB at PP hard)


def dump_outputs(path, tr, t):
    """Write what the rollout handed its caller in its last lock-step iteration (record index t) as <path>/<name>.npy:
    the RolloutBatch fields of that iteration and the merged statistics vector in full, the LSTM state (h, c) for a
    fixed seeded sample of env slots.  float32 (integers and masks are exact in it), float64 for the statistics."""
    import numpy as np
    import torch
    b, B, N = tr._buf, tr.env.env.nenvs, tr.args.nagents
    out = dict(action=b["action"][t], logp=b["logp"][t], value=b["value"][t].view(B, N), reward=b["reward"][t],
               episode_mask=b["emask"][t], episode_mini_mask=b["mini"][t], alive_mask=b["ralive"][t],
               valid=b["valid"][t])
    slots = np.sort(np.random.default_rng(0).choice(B, size=min(B, HIDDEN_SAMPLE_SLOTS), replace=False))
    idx = torch.as_tensor(slots, device=b["h"].device)
    out.update(h=b["h"].view(B, N, -1)[idx], c=b["c"].view(B, N, -1)[idx])
    os.makedirs(path, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(path, k + ".npy"), v.float().cpu().numpy())
    np.save(os.path.join(path, "stat.npy"), b["statvec"].cpu().numpy())


def train_leg(opts, build, MultiGPUTrainer, world, dev, dist, torch):
    """agent-env-steps/s of complete training updates: every rank runs MultiGPUTrainer.train_batch (rollout with
    the reference batch boundary, compute_grad, ONE all-reduce of the flat gradient buffer + the statistics vector,
    RMSprop) -- the like-for-like of the reference's MultiProcessTrainer.train_batch."""
    a, env, net, tr = build("index", opts.train_envs or None, record_for_grad=True, batch_size=opts.train_batch_size,
                            grad_impl=opts.grad_impl, batch_boundary=opts.train_boundary, value_coeff=0.01, entr=0.0, gamma=1.0, normalize_rewards=False,
                            detach_gap=10000, grad_window=opts.grad_window)
    mgt = MultiGPUTrainer(a, lambda: tr)
    N = a.nagents
    mgt.train_batch(0)                                        # warm-up (allocations, graph-free)
    torch.cuda.synchronize()
    times, steps, phases = [], 0, []
    for u in range(opts.train_updates):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        stat = mgt.train_batch(u + 1)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        times.append(float(t.item()))
        steps += int(stat["num_steps"])                       # already summed over ranks
    # split of one update on this rank: rollout alone vs the rest
    torch.cuda.synchronize()
    T, quota = tr.batch_plan()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    tr.rollout(T, 0, quota=quota)
    e1.record()
    torch.cuda.synchronize()
    roll_ms = e0.elapsed_time(e1)
    tot_ms = sum(times)
    return dict(value=steps * N / (tot_ms * 1e-3), unit="agent-env-steps/s", updates=opts.train_updates,
                envs_per_gpu=a.nenvs, batch_size=a.batch_size, lock_steps_per_update=T,
                ms_per_update=tot_ms / opts.train_updates, rollout_ms=roll_ms,
                grad_reduce_step_ms=tot_ms / opts.train_updates - roll_ms, grad_impl=tr.grad_impl,
                replica_max_abs_diff=mgt.replica_checksum(), collectives_per_update=mgt.collectives / max(1, opts.train_updates + 1)
                if world > 1 else 0,
                api="MultiGPUTrainer.train_batch (all ranks; device time, max over ranks)")


def trainer_api_leg(opts, build, world, dev, dist, torch, calls=2):
    """The call a reference user makes for a rollout (main.py -> Trainer.run_batch, trainer.py:227-242), end to end:
    ``batch, stat = Trainer.run_batch(epoch)`` with the reference batch boundary, then EVERY array of the returned
    batch copied to pinned host memory (the reference hands its batch back as host data), wall clock, max over ranks.
    Reported beside the per-step host loop (which stays the e2e headline: it crosses the PCIe bus twice per step)."""
    a, env, net, tr = build("index", None, batch_size=opts.train_batch_size, batch_boundary=opts.train_boundary,
                            use_graph=not opts.no_graph)
    N = a.nagents
    batch, stat = tr.run_batch(0)                             # warm-up: buffers, graph capture
    host = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in batch._asdict().items()}
    nbytes = sum(v.numel() * v.element_size() for v in host.values())
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    steps = 0
    t0 = time.perf_counter()
    for k in range(calls):
        batch, stat = tr.run_batch(k + 1)                     # includes the stat vector's device->host copy
        for f, v in batch._asdict().items():
            host[f].copy_(v, non_blocking=True)
        torch.cuda.synchronize()
        steps += int(stat["num_steps"])
    dt = time.perf_counter() - t0
    agg = torch.tensor([dt, float(steps)], device=dev, dtype=torch.float64)
    if world > 1:
        mx, sm = agg.clone(), agg.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dt, steps = float(mx[0].item()), float(sm[1].item())
    T = tr.batch_plan()[0]
    return dict(value=steps * N / dt, unit="agent-env-steps/s", calls=calls, lock_steps_per_call=T,
                ms_per_call=1e3 * dt / calls, d2h_bytes_per_call=nbytes * world, d2h_bytes_per_step=nbytes * world // T,
                api="Trainer.run_batch (reference batch boundary, batch_size %d) + every array of the returned batch "
                    "copied to pinned host memory; wall clock, max over ranks" % a.batch_size)


def per_kernel_times(tr, a, env, net, steps, C, torch, _lib):
    """Average device time of each kernel of the step, CUDA events around every launch."""
    lib = _lib.load()
    e, b = env.env, tr._buf
    B = e.nenvs
    cfg = net.policy_cfg(B)
    cfg.seed, cfg.env_id0 = e.cfg.seed, e.cfg.env_id0
    w = net.packed()
    s = _lib.stream()
    is_tj = a.env_name == "traffic_junction"
    hard = int(bool(a.hard_attn))
    nh = len(a.naction_heads)
    ev, split = {}, {}

    def timed(name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        _lib.check(fn())
        e1.record()
        ev.setdefault(name, []).append((e0, e1))

    ws = net.workspace(B)[0]
    W_ = 2 * e.vision + 1
    fused_x = tr._fused_x()                                   # index encoder fused into the policy step
    src = {}
    if fused_x:
        src = dict(tj_env=C.addressof(e.cfg), tj_state=C.addressof(e.state)) if is_tj else \
            dict(pp_env=C.addressof(e.cfg), pp_state=C.addressof(e.state))
        src["x_table"] = _lib.ptr(tr._encoder_table(cfg, w))  # same path as Trainer._enqueue
    for t in range(steps):
        if tr.obs_mode == "dense":
            if is_tj:
                timed("obs_gather", lambda: lib.ic3_tj_obs(C.byref(e.cfg), C.byref(e.state), b["obs"].data_ptr(), s))
            else:
                timed("obs_gather", lambda: lib.ic3_pp_obs(C.byref(e.cfg), C.byref(e.state), b["obs"].data_ptr(), s))
            timed("encoder_dense", lambda: lib.ic3_encoder_dense(C.byref(cfg), C.byref(w), b["obs"].data_ptr(),
                                                                 b["x"].data_ptr(), s))
        elif fused_x:
            pass
        elif is_tj:
            timed("encoder_index", lambda: lib.ic3_tj_encoder_index(C.byref(e.cfg), C.byref(e.state), C.byref(cfg),
                                                                    C.byref(w), b["x"].data_ptr(), s))
        else:
            timed("encoder_index", lambda: lib.ic3_pp_encoder_index(C.byref(e.cfg), C.byref(e.state), C.byref(cfg),
                                                                    C.byref(w), b["x"].data_ptr(), s))
        io = _lib.PolicyIO(x=None if fused_x else b["x"].data_ptr(), h=b["h"].data_ptr(), c=b["c"].data_ptr(),
                           comm_action=b["comm"].data_ptr() if hard else None, alive=b["alive"].data_ptr(),
                           fresh=b["fresh"].data_ptr(), tick=e.tick.data_ptr(), draws=None, h_out=b["h"].data_ptr(),
                           c_out=b["c"].data_ptr(), value=b["value"][t].data_ptr(), logp=b["logp"][t].data_ptr(),
                           action=b["action"][t].data_ptr(), workspace=_lib.ptr(ws),
                           err=b["err"].data_ptr(), **src)
        timed("policy_step", lambda: lib.ic3_policy_step(C.byref(cfg), C.byref(w), C.byref(io), s))
        if net.policy_impl == "tc" and t >= steps - 4:        # split of the last few steps (extra passes, same state)
            ms3 = (C.c_float * 3)()
            _lib.check(lib.ic3_policy_step_profile(C.byref(cfg), C.byref(w), C.byref(io), s, ms3))
            for nm, v in zip(("prep", "lstm_tc", "heads_finish"), ms3):
                split.setdefault(nm, []).append(float(v))
        r = _lib.RolloutIO(t=t, max_steps=a.max_steps, nheads=nh, hard_attn=hard,
                           comm_action_one=int(bool(a.comm_action_one)), last=0, action=b["action"][t].data_ptr(),
                           t_ep=b["t_ep"].data_ptr(), fresh=b["fresh"].data_ptr(), comm_next=b["comm"].data_ptr(),
                           alive_next=b["alive"].data_ptr(), rec_reward=b["reward"].data_ptr(),
                           rec_episode_mask=b["emask"].data_ptr(), rec_mini_mask=b["mini"].data_ptr(),
                           rec_alive=b["ralive"].data_ptr(), stat_reward=b["stat_reward"].data_ptr(),
                           stat_comm=b["stat_comm"].data_ptr(), stat_success=b["stat_success"].data_ptr(),
                           stat_episodes=b["stat_episodes"].data_ptr(), stat_steps=b["stat_steps"].data_ptr())
        if is_tj:
            timed("env_step", lambda: lib.ic3_tj_step(C.byref(e.cfg), C.byref(e.state), b["action"][t].data_ptr(), nh,
                                                      None, b["step_reward"].data_ptr(), None, b["err"].data_ptr(),
                                                      C.byref(r), s))
        else:
            timed("env_step", lambda: lib.ic3_pp_step(C.byref(e.cfg), C.byref(e.state), b["action"][t].data_ptr(), nh,
                                                      b["step_reward"].data_ptr(), None, b["err"].data_ptr(),
                                                      C.byref(r), s))
    torch.cuda.synchronize()
    out = {k: sum(x.elapsed_time(y) for x, y in v) / len(v) for k, v in ev.items()}
    out.update({k: sum(v) / len(v) for k, v in split.items()})
    return out


def e2e_loop(a, env, net, steps, np, torch, select_action):
    """The reference-shaped call sequence of Trainer.get_episode (trainer.py:43-108) with HOST arrays for
    everything the reference keeps in numpy (actions, comm_action, alive_mask, reward, done); observations
    and hidden states stay in HBM.  Pinned host buffers; every step synchronises like the reference does."""
    B, N = a.nenvs, a.nagents
    nh = len(a.naction_heads)
    is_tj = a.env_name == "traffic_junction"
    e = env.env
    e.strict = False
    pin = lambda *s, dtype: torch.empty(*s, dtype=dtype).pin_memory()
    from ic3net_b200.action_utils import translate_action
    act_h = [pin(B, N, dtype=torch.int32) for _ in range(nh)]           # per-head host arrays, like translate_action's
    rew_h, done_h = pin(B, N, dtype=torch.float32), pin(B, dtype=torch.bool)
    alive_h = pin(B, N, dtype=torch.uint8)
    comm_h = pin(B, N, dtype=torch.uint8)
    ones_h = torch.ones(B, N, dtype=torch.uint8)
    h2d = d2h = 0

    phases = dict(policy_enqueue=0.0, wait_actions=0.0, env_enqueue=0.0, wait_reward=0.0)

    def one_step(obs, hc, info, count):
        nonlocal h2d, d2h
        t0 = time.perf_counter()
        action_out, value, hc = net([obs, hc], info)                     # comm_action / alive_mask: host -> device
        action = select_action(a, action_out)
        heads_d, _actual = translate_action(a, env, action)              # per-head arrays (trainer.py:65-66)
        for k in range(nh):
            act_h[k].copy_(heads_d[k], non_blocking=True)                # D2H (the reference's .numpy())
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        obs, reward, done, info_env = env.step(act_h)                    # H2D actions (the wrapper passes head 0)
        rew_h.copy_(reward, non_blocking=True)                           # D2H
        done_h.copy_(done, non_blocking=True)
        t3 = time.perf_counter()
        nxt = {}
        if a.hard_attn:
            comm_h.copy_(act_h[-1] if not a.comm_action_one else ones_h)    # trainer.py:55-58, on the host
            nxt["comm_action"] = comm_h
        if is_tj:
            alive_h.copy_(info_env["alive_mask"], non_blocking=True)     # D2H
            nxt["alive_mask"] = alive_h
        torch.cuda.synchronize()
        if count:
            t4 = time.perf_counter()
            for k, v in zip(("policy_enqueue", "wait_actions", "env_enqueue", "wait_reward"),
                            (t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
                phases[k] += v
            h2d += act_h[0].numel() * 4 + (comm_h.numel() if a.hard_attn else 0) + (alive_h.numel() if is_tj else 0)
            d2h += nh * act_h[0].numel() * 4 + rew_h.numel() * 4 + done_h.numel() + (alive_h.numel() if is_tj else 0)
        if not is_tj and bool(done_h.any()):                             # finished PP envs start a new episode
            m = done_h.to(torch.uint8)
            e.reset(mask=m, want_obs=False)
            obs = env._flatten_obs(e._obs_handle() if e.obs_api == 'handle' else e._get_obs())
            keep = (~done_h).to(obs.device).repeat_interleave(N).unsqueeze(1).float()
            hc = (hc[0] * keep, hc[1] * keep)
            if a.hard_attn:
                comm_h.mul_((~done_h).to(torch.uint8).unsqueeze(1))
        return obs, hc, nxt

    obs = env.reset(0)
    hc = net.init_hidden(B)
    info = {"comm_action": torch.zeros(B, N, dtype=torch.uint8).pin_memory()} if a.hard_attn else {}
    for _ in range(3):
        obs, hc, info = one_step(obs, hc, info, False)
    torch.cuda.synchronize()
    import gc
    gc.collect()
    gc.freeze()          # keep the generational GC from walking the whole (torch-sized) heap inside the timed loop
    ms0 = torch.cuda.memory_stats()
    t0 = time.perf_counter()
    per_step = []
    for _ in range(steps):
        ts = time.perf_counter()
        obs, hc, info = one_step(obs, hc, info, True)
        per_step.append(time.perf_counter() - ts)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    gc.unfreeze()
    per_step.sort()
    ms1 = torch.cuda.memory_stats()
    e.err.zero_()
    return dict(value=B * N * steps / dt, unit="agent-env-steps/s", seconds=dt, h2d_bytes_per_step=h2d // steps,
                d2h_bytes_per_step=d2h // steps, steps=steps, ms_per_step=1e3 * dt / steps,
                phases_ms={k: round(1e3 * v / steps, 4) for k, v in phases.items()},
                step_ms_median=round(1e3 * per_step[len(per_step) // 2], 4), step_ms_max=round(1e3 * per_step[-1], 4),
                step_ms_sorted_tail=[round(1e3 * x, 3) for x in per_step[-4:]],
                cuda_mallocs_in_loop=int(ms1.get("num_device_alloc", 0) - ms0.get("num_device_alloc", 0)),
                cuda_frees_in_loop=int(ms1.get("num_device_free", 0) - ms0.get("num_device_free", 0)),
                api="GymWrapper.reset/step (observation %s) -> CommNetMLP.forward -> select_action -> host actions -> "
                    "GymWrapper.step -> host reward/done" % ("handle" if e.obs_api == "handle" else "tensor"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="pp_hard_ic3net", choices=sorted(WORKLOADS))
    ap.add_argument("--obs_mode", default="dense", choices=["dense", "index"])
    ap.add_argument("--policy_impl", default=None, choices=["tc", "simt"],
                    help="tcgen05 tensor-core policy kernels (default for hid_size 128) or the fp32 SIMT kernel")
    ap.add_argument("--no_graph", action="store_true",
                    help="enqueue every kernel of the rollout eagerly (default: CUDA-graph replay of the K-step region, "
                         "what Trainer(use_graph=True) does; removes the host launch skew between ranks)")
    ap.add_argument("--graph", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--train_updates", type=int, default=2, help="timed MultiGPUTrainer.train_batch updates (0 = skip)")
    ap.add_argument("--train_envs", type=int, default=0, help="env slots per GPU of the train_batch leg (0 = workload's)")
    ap.add_argument("--train_batch_size", type=int, default=500, help="--batch_size of the train_batch leg (reference default)")
    ap.add_argument("--grad_impl", default="auto", choices=["auto", "autograd", "manual", "kernels"],
                    help="compute_grad implementation of the train_batch leg (auto = the Trainer default: the BPTT kernels)")
    ap.add_argument("--train_boundary", default="reference", choices=["reference", "cut"])
    ap.add_argument("--grad_window", type=int, default=40)
    ap.add_argument("--quick", action="store_true", help="skip the e2e / index / CPU / train legs (profiling runs)")
    ap.add_argument("--skip", default="", help="comma list of legs to skip: train,e2e,kernels,index,cpu")
    ap.add_argument("--obs_chunk_mb", type=float, default=0.0,
                    help="dense rollout: gather + encode observations in chunks of env slots of at most this size "
                         "(experiment; 0 = the whole batch at once, the measured optimum)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed (rank 0's env slots) as "
                         "DIR/<name>.npy; the same arguments give the same inputs on every run")
    opts = ap.parse_args()
    if opts.dump_outputs and opts.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 implementation")
    if opts.impl == "reference":
        return reference_arm(opts)
    return gpu_arm(opts)


if __name__ == "__main__":
    sys.exit(main())
