"""bench.py -- optimizer steps/s of the DotaClient optimizer hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c1] [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, NCCL)

``--dump-outputs DIR`` writes what the last timed train() step handed its caller (rank 0) as DIR/<name>.npy: the loss
terms, per-head entropies and grad norms it returns, and the policy parameters it updated (see ``step_outputs``).  Inputs
and initial weights are seeded, so two builds run with the same arguments can be compared output for output.

A "step" is one ``DotaOptimizer.train()`` call (forward, PPO loss, backward, gradient all-reduce, clip, Adam)
on one synthetic experience batch.  Default workload = BASELINE.json configs[1] ("c2": batch 256 x seq 512,
hidden 128, LSTM) PER GPU (weak scaling); ``value`` counts one such batch per GPU per step.

Keys: value (inputs resident in HBM), e2e (inputs in pinned host memory, H2D + result D2H inside the timed
region), roofline (recurrence fwd+bwd kernels: algorithmic bytes / CUDA-event time / measured HBM peak),
cpu_baseline (the oracle port of the reference's train() on the host cores, bounded sample), clocks,
gpu_launches.  ``--impl reference`` times the reference's CPU implementation (oracle port; the reference is
pure Python + torch CPU and cannot travel to the GPU box) on the same config.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIGS = {                       # BASELINE.json configs; batch is PER GPU
    "c1": dict(batch=1, seq_len=64, hidden=128, cell="lstm"),
    "c2": dict(batch=256, seq_len=512, hidden=128, cell="lstm"),
    "c3": dict(batch=512, seq_len=512, hidden=256, cell="lstm"),
    "c4": dict(batch=512, seq_len=1024, hidden=512, cell="lstm"),
    # configs[4]: 40-agent replay stream through the in-process broker, the reference's own defaults
    # (optimizer.py:781-786: min_seq_per_epoch 1024, seq_len 16, epochs 4; policy.py:66: 256-wide GRU)
    "c5": dict(batch=1024, seq_len=16, hidden=256, cell="gru", stream=True),
}
FALLBACK_HBM_GBS = 6650.0         # /opt/skills/guides/B200_PROFILING.md fallback


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--config", choices=sorted(CONFIGS), default="c2")
    p.add_argument("--cell", choices=["gru", "lstm"], default=None)
    p.add_argument("--batch", type=int, default=None)
    p.add_argument("--seq-len", type=int, default=None)
    p.add_argument("--hidden", type=int, default=None)
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cuda-profiler", action="store_true",
                   help="bracket the HBM-resident timed region with cudaProfilerStart/Stop (for ncu --profile-from-start off)")
    p.add_argument("--skip-e2e", action="store_true", help="(profiling only) skip the host-buffer timed region")
    p.add_argument("--no-extra", action="store_true", help="skip the extra_configs block (C1/C3/C4 per-GPU shapes, 3 steps each)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the outputs of the last timed step as DIR/<name>.npy (GPU train() arm only)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be >= 1")
    if args.dump_outputs is not None and (args.impl == "reference" or CONFIGS[args.config].get("stream")):
        p.error("--dump-outputs applies to the GPU train() arm, not to --impl reference or the stream config")
    return args


def resolve_config(args):
    cfg = dict(CONFIGS[args.config])
    for k, a in (("batch", args.batch), ("seq_len", args.seq_len), ("hidden", args.hidden), ("cell", args.cell)):
        if a is not None:
            cfg[k] = a
    return cfg


def measured_peak_hbm():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ CPU baseline
def log(msg):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sys.stderr.write("[bench %.1fs] %s\n" % (time.perf_counter() - _T0, msg))
    sys.stderr.flush()


_T0 = time.perf_counter()


def usable_cores():
    """Cores this process may actually use: affinity mask, capped by the cgroup CPU quota if there is one."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except Exception:
        pass
    return n


def cpu_reference_steps_per_sec(cfg, budget_s=20.0, threads=None):
    """The oracle port of the reference's ``DotaOptimizer.train`` (optimizer.py:581-689) on the host cores.

    Bounded sample: ``b`` sequences of the config's seq_len/hidden/cell; ``b`` starts at 1 and doubles until one
    step takes >= 1 s (or b reaches the config's batch), then steps are timed for ~budget_s.  steps/s for the full
    batch is extrapolated linearly in the batch size (the work is per-token).
    """
    import torch
    from oracle import ref_optimizer as RO
    from oracle.ref_policy import RefPolicy
    from dotaclient_b200.synthetic import make_rollout
    cores = threads or min(usable_cores(), 64)            # torch CPU stops scaling on these GEMM sizes long before 64
    torch.set_num_threads(cores)
    S, H, cell, B = cfg["seq_len"], cfg["hidden"], cfg["cell"], cfg["batch"]
    torch.manual_seed(7)
    opt = RO.RefOptimizer(RefPolicy(H, cell), seq_len=S)
    seqs = opt.experiences_from_rollout(make_rollout(S, 7))
    opt.train(seqs)                                        # untimed warm-up (a cold first call must not end the sizing loop)
    b = 1
    t_begin = time.perf_counter()
    while True:
        t0 = time.perf_counter()
        opt.train(seqs)
        dt = time.perf_counter() - t0
        if dt >= 1.0 or b >= B or b >= 32 or time.perf_counter() - t_begin > budget_s / 2:
            break
        for i in range(b):
            seqs.extend(opt.experiences_from_rollout(make_rollout(S, 7 + b + i)))
        b *= 2
    t0, n = time.perf_counter(), 0
    while True:
        opt.train(seqs)
        n += 1
        el = time.perf_counter() - t0
        if el > budget_s / 2 or n >= 20:
            break
    b = len(seqs)
    sample_steps_per_s = n / el
    full = sample_steps_per_s * b / B
    sample = "oracle port of optimizer.py:581-689, batch %d x seq %d (hidden %d, %s), %d steps in %.1f s on %d threads; " \
             "scaled x%d/%d to batch %d" % (b, S, H, cell, n, el, cores, b, B, B)
    return full, cores, sample, b


def run_reference_arm(args, cfg):
    """``--impl reference``: the reference's CPU ``train()`` (oracle port: the reference is pure Python + torch CPU and
    cannot travel to the GPU box) on the host cores, same config/metric.  Each step is one train() on a bounded sample
    (``b`` of the config's ``batch`` sequences, full seq_len); steps/s is scaled by b/batch.  Rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from oracle import ref_optimizer as RO
    from oracle.ref_policy import RefPolicy
    from dotaclient_b200.synthetic import make_rollout
    cores = min(usable_cores(), 64)
    torch.set_num_threads(cores)
    S, H, cell, B = cfg["seq_len"], cfg["hidden"], cfg["cell"], cfg["batch"]
    torch.manual_seed(7)
    opt = RO.RefOptimizer(RefPolicy(H, cell), seq_len=S)
    seqs = opt.experiences_from_rollout(make_rollout(S, 7))
    opt.train(seqs)                                        # untimed: thread pool / allocator warm-up must not end the sizing loop
    b = 1
    while True:                                            # grow the sample until one step takes >= 1 s (cap 32 sequences)
        t0 = time.perf_counter()
        opt.train(seqs)
        if time.perf_counter() - t0 >= 1.0 or b >= B or b >= 32:
            break
        for i in range(b):
            seqs.extend(opt.experiences_from_rollout(make_rollout(S, 7 + b + i)))
        b *= 2
    b = len(seqs)
    for _ in range(args.warmup):
        opt.train(seqs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        opt.train(seqs)
    el = time.perf_counter() - t0
    value = args.steps / el * b / B
    sample = "oracle port of optimizer.py:581-689, batch %d x seq %d (hidden %d, %s), %d steps in %.1f s on %d threads; " \
             "scaled x%d/%d to batch %d" % (b, S, H, cell, args.steps, el, cores, b, B, B)
    line = {
        "impl": "reference", "metric": "optimizer_steps_per_sec", "value": value, "unit": "steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(cfg, args.gpus, "cpu"),
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample,
                         "sample_batch": b, "scale_factor": b / float(B)},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "ONE CPU process on this host's cores (rank 0 only), also when --gpus N > 1: N reference ranks would share the same "
                "cores, so the per-rank-batch rate does not grow with N; a ratio against it at N GPUs compares N GPUs with one host",
    }
    emit(line)


def workload_config(cfg, n_gpus, where):
    return {"workload": "BASELINE configs: synthetic experience batch=%d seq=%d hidden=%d per GPU, %s cell; "
                        "one DotaOptimizer.train() per step" % (cfg["batch"], cfg["seq_len"], cfg["hidden"], cfg["cell"]),
            "batch_per_gpu": cfg["batch"], "global_batch": cfg["batch"] * n_gpus, "seq_len": cfg["seq_len"],
            "hidden": cfg["hidden"], "cell": cfg["cell"], "parallelism": "dp%d" % n_gpus,
            "l2": "per-step inputs exceed the 126 MB L2" if cfg["batch"] * cfg["seq_len"] * 2100 > 126e6
                  else "working set below the 126 MB L2 (stated, not flushed: C1 is the reference's latency case)"}


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:                                         # reaped here, so that no sampler outlives the run
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ GPU arm
def run_stream(args, cfg):
    """BASELINE configs[4]: 40 agents (threads) publish pickled rollouts of 1000-1400 steps into the in-process
    ``MessageQueue``; every rank runs ``DotaOptimizer.run_iteration`` (pull -> prep -> epochs x train -> publish) and
    steady-state optimizer steps/s is reported.  Secondary configuration (not the headline bench line)."""
    import pickle
    import random
    import torch
    import torch.distributed as dist
    from dotaclient_b200.optimizer import DotaOptimizer, MessageQueue
    from dotaclient_b200.synthetic import make_rollout
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl")
    epochs = 4
    opt = DotaOptimizer(rmq_host="stream", rmq_port=rank, epochs=epochs, min_seq_per_epoch=cfg["batch"], seq_len=cfg["seq_len"],
                        learning_rate=5e-5, checkpoint=False, pretrained_model=None, mq_prefetch_count=1,
                        log_dir=tempfile.mkdtemp(), entropy_coef=5e-4, vf_coef=0.5, run_local=True,
                        hidden_size=cfg["hidden"], cell=cfg["cell"], rollout_prefetch=16)
    agents = max(1, 40 // world)
    rng = random.Random(7 + rank)
    pool = [pickle.dumps(make_rollout(rng.randint(1000, 1400), 7 + 1000 * rank + i, with_canvas=True)) for i in range(8)]
    stop = threading.Event()
    mq = MessageQueue(host="stream", port=rank, prefetch_count=1, use_model_exchange=False)
    mq.connect()

    def agent(i):
        j = i
        while not stop.is_set():
            if mq.xp_queue_size < 64:
                mq.publish_experience(pool[j % len(pool)])
                j += 1
            else:
                time.sleep(0.001)
    threads = [threading.Thread(target=agent, args=(i,), daemon=True) for i in range(agents)]
    for th in threads:
        th.start()
    for it in range(1, 1 + max(1, args.warmup)):
        opt.run_iteration(it)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    env_steps = 0
    for it in range(args.steps):
        m = opt.run_iteration(100 + it)
        env_steps += int(round(m[opt.SPEED_KEY] * m["timing/it"]))
    torch.cuda.synchronize()
    el = torch.tensor([time.perf_counter() - t0], device="cuda")
    if world > 1:
        dist.all_reduce(el, op=dist.ReduceOp.MAX)
    stop.set()
    if rank == 0:
        sec = float(el.item())
        emit({"metric": "optimizer_steps_per_sec", "value": world * args.steps * epochs / sec, "unit": "steps/s",
                          "n_gpus": world, "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": 1000 * sec / (args.steps * epochs),
                          "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                          "env_steps_per_sec": world * env_steps / sec,
                          "config": {"workload": "BASELINE configs[4]: 40-agent replay stream, in-process broker, reference defaults "
                                                 "(>=1024 seqs x 16 per iteration, 4 epochs, hidden 256 GRU); 'step' = one train() call "
                                                 "including its share of experience prep", "agents": agents * world,
                                     "parallelism": "dp%d" % world}})
    opt.close()
    finish_process(world)


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of this run, on the process's real stdout."""
    out = os.fdopen(os.dup(_REAL_STDOUT), "w") if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def algorithmic_rnn_bytes(cfg):
    G = 4 if cfg["cell"] == "lstm" else 3
    return 12.0 * cfg["batch"] * cfg["seq_len"] * (G + 1) * cfg["hidden"]          # SURVEY.md 8(d): fwd + bwd


def build_optimizer(cfg, rank):
    from dotaclient_b200.optimizer import DotaOptimizer
    return DotaOptimizer(rmq_host="bench", rmq_port=rank, epochs=1, min_seq_per_epoch=cfg["batch"], seq_len=cfg["seq_len"],
                         learning_rate=5e-5, checkpoint=False, pretrained_model=None, mq_prefetch_count=1, log_dir=tempfile.mkdtemp(),
                         entropy_coef=5e-4, vf_coef=0.5, run_local=True, hidden_size=cfg["hidden"], cell=cfg["cell"])


def measure_prep(opt, rollouts, repeats=2):
    """Experience prep of one iteration through the product's batched path (optimizer.py:328-430 for all rollouts at once):
    host numpy rollouts -> H2D -> encoder -> recurrence -> heads -> selected log-probs -> segmented GAE -> stacked batch.
    Returns (batch, wall ms of the last repeat, per-kernel CUDA-event ms of the last repeat)."""
    import torch
    from dotaclient_b200 import ops
    batch, ms, kern = None, 0.0, {}
    for _ in range(repeats):
        del batch
        torch.cuda.synchronize()
        ops.PROFILE.reset(enabled=True)
        t0 = time.perf_counter()
        with torch.no_grad():
            batch = opt.batch_from_rollouts(rollouts)
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        kern = ops.PROFILE.summary(1)
        ops.PROFILE.reset(enabled=False)
    return batch, ms, kern


DUMP_MAX_ELEMENTS = 1 << 21       # larger arrays are dumped as a fixed seeded sample of this many elements
DUMP_MAX_BYTES = 64 << 20


def step_outputs(opt, result):
    """What one train() call hands its caller, as host arrays named for --dump-outputs: the loss terms, per-head entropies and
    grad norms it returns, and the policy parameters it updates in place.  An array of more than DUMP_MAX_ELEMENTS elements
    (recurrent weights of cells far wider than the BASELINE ones) is replaced by its flattened values at the sorted positions
    np.random.default_rng(0).choice(n, DUMP_MAX_ELEMENTS, replace=False), the same in every run and every build."""
    import numpy as np
    losses, entropies, norms = result
    named = dict(losses)
    named.update(("entropy." + k, v) for k, v in entropies.items())
    named.update(("grad_norm." + k, v) for k, v in norms.items())
    named.update(("param." + k, v) for k, v in opt.policy_base.state_dict().items())
    out = {}
    for name, v in named.items():
        a = v.detach().cpu().numpy()
        if a.size > DUMP_MAX_ELEMENTS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))]
        out[name] = a
    assert sum(a.nbytes for a in out.values()) <= DUMP_MAX_BYTES
    return out


def measure_config(cfg, args, world, rank, dev, steps, warmup, with_e2e, dump=False):
    """One BASELINE configuration on this rank's GPU: prep, `steps` timed train() calls (inputs resident in HBM), optional
    end-to-end loops from pinned host memory.  Returns a dict of raw measurements (rank-local except the max-over-ranks ms);
    with ``dump``, ``outputs`` holds ``step_outputs`` of the last timed step."""
    import torch
    import torch.distributed as dist
    from dotaclient_b200 import ops
    from dotaclient_b200.synthetic import make_rollout, rollout_seed
    B, S = cfg["batch"], cfg["seq_len"]
    opt = build_optimizer(cfg, rank)
    log("[%s] optimizer built; generating %d rollouts of %d steps" % (cfg["name"], B, S))
    rollouts = [make_rollout(S, rollout_seed(rank, i)) for i in range(B)]
    batch_dev, prep_ms, prep_kern = measure_prep(opt, rollouts)
    del rollouts
    log("[%s] prep %.1f ms (batched, incl. H2D of the raw rollouts)" % (cfg["name"], prep_ms))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    enqueue, last = [], [None]

    def step_dev():
        last[0] = opt.train(batch_dev)
        enqueue.append(opt.host_enqueue_s)

    for _ in range(max(3, warmup)):
        step_dev()
    # (1) the headline: train() on a device-resident batch -- after the warm-up the step replays from its CUDA graph
    if args.cuda_profiler:
        torch.cuda.profiler.start()
    ms_total = timed(step_dev, steps)
    if args.cuda_profiler:
        torch.cuda.profiler.stop()
    enq = 1e3 * sum(enqueue[-steps:]) / steps
    graphed = any(isinstance(v, tuple) for v in opt._graphs.values())
    outputs = step_outputs(opt, last[0]) if dump else None      # before the steps below move the parameters on
    # (2) the same steps launch by launch with CUDA events around every C-ABI call: the per-kernel table of the roofline
    ops.PROFILE.reset(enabled=True)
    step_dev()                                  # untimed: the launch-by-launch path re-grows its allocator pool after the capture
    ops.PROFILE.reset(enabled=True)
    ms_eager = timed(step_dev, steps)
    prof = ops.PROFILE.summary(steps)
    prof_bytes = {k: v / steps for k, v in ops.PROFILE.bytes.items()}
    launches = ops.PROFILE.launches
    ops.PROFILE.reset(enabled=False)
    out = {"ms_per_step": ms_total / steps, "ms_per_step_launch_by_launch": ms_eager / steps, "cuda_graph": graphed,
           "prep_ms": prep_ms, "prep_kernels": prep_kern, "kernels": prof, "kernel_bytes": prof_bytes,
           "launches": launches, "host_enqueue_ms": enq, "host_enqueue_ms_launch_by_launch": 1e3 * sum(enqueue[-steps:]) / steps,
           "h2d_bytes": batch_dev.nbytes(), "outputs": outputs}
    log("[%s] timed region (HBM-resident): %.2f ms/step" % (cfg["name"], out["ms_per_step"]))
    if with_e2e:
        batch_host = batch_dev.pin_memory()
        seqs_host = None
        step_serial = lambda: opt.train(batch_host)  # noqa: E731   (upload, then compute)
        pending = []

        def step_e2e():
            # double-buffered upload through the public API: step k+1's inputs start their H2D copy (from pinned host memory)
            # before step k is launched, so the transfer runs next to step k's kernels; every timed step performs one full upload
            cur = pending.pop() if pending else opt.prefetch(batch_host)
            pending.append(opt.prefetch(batch_host))
            opt.train(cur)

        for _ in range(2):
            step_serial()
        out["ms_e2e_serial"] = timed(step_serial, steps) / steps
        for _ in range(5):                          # both input slots seen once (launch by launch) and captured once
            step_e2e()
        out["ms_e2e"] = timed(step_e2e, steps) / steps
        pending.clear()
        # the reference's own call signature: train(list_of_Sequence) with device-resident records, as its
        # experiences_from_rollout leaves them (:355-363) -- the list is re-stacked on every call like :587-615
        if B <= 512:
            seqs_host = sequences_of(batch_dev)
            for _ in range(2):
                opt.train(seqs_host)
            out["ms_e2e_list_api"] = timed(lambda: opt.train(seqs_host), steps) / steps
        log("[%s] timed region (e2e): %.2f ms/step" % (cfg["name"], out["ms_e2e"]))
        del batch_host, seqs_host
    opt.close()                                 # captured graphs (with NCCL work when data-parallel) go before the process group does
    del batch_dev, opt
    torch.cuda.empty_cache()
    return out


def sequences_of(batch):
    """The stacked batch as the reference's ``list`` of per-sequence records (views of the device batch)."""
    from dotaclient_b200.optimizer import Sequence
    out = []
    for b in range(batch.batch_size):
        hid = (batch.h0[:, b:b + 1], batch.c0[:, b:b + 1]) if batch.c0 is not None else batch.h0[:, b:b + 1]
        s = Sequence(game_id=0, weight_version=1, team_id=2, observations={k: v[:, b] for k, v in batch.observations.items()},
                     actions={k: v[:, b] for k, v in batch.actions.items()}, masks={k: v[:, b] for k, v in batch.masks.items()},
                     values=None, rewards=None, hidden=hid, old_logp=batch.old_logp[:, b])
        s.advantages, s.returns = batch.advantages[:, b], batch.returns[:, b]
        out.append(s)
    return out


def kernel_table(meas, peak):
    table = {}
    for name, ms in meas["kernels"].items():
        nbytes = meas["kernel_bytes"].get(name, 0)
        gbps = (nbytes / (ms * 1e-3) / 1e9) if ms > 0 else 0.0
        table[name] = {"ms": ms, "bytes": nbytes, "GBps": gbps, "frac": gbps / peak}
    return table


KERNEL_FAMILIES = {   # label -> (profile-span names, key of profiles/kernel_traffic.json)
    "tcgen05 3xTF32 GEMM, forward + data gradient (dc_gemm_tf32x3*, dc_gemm_unit_max)": (["gemm_tf32x3", "gemm_unit_max"], "gemm_fwd_dgrad"),
    "tcgen05 3xTF32 weight-gradient GEMM (dc_gemm_wgrad_tf32x3*, dc_unit_wgrad_routed)": (["gemm_wgrad"], "gemm_wgrad"),
    "fused unit-encoder data gradient (dc_unit_dgrad_fused: generated d_emb x W_g on tcgen05 3xTF32, ReLU mask + dW_b reduction in the epilogue)":
        (["unit_dgrad_fused"], "unit_dgrad_fused"),
    "recurrence fwd+bwd (dc_rnn_seq_fwd + dc_rnn_seq_bwd)": (["rnn_fwd", "rnn_bwd"], "rnn"),
}


def measured_peak_tf32():
    """Dense tf32 tensor peak = half the measured dense bf16 rate (sustained figure: the kernel runs inside a long step)."""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            rec = json.load(f)
        return float(rec.get("bf16_tflops_sustained", rec["bf16_tflops"])) / 2.0, "measured bf16 sustained / 2 (MEASURED_PEAKS.json)"
    except Exception:
        return 2250.0 / 2.0, "nominal dense bf16 / 2 (B200_PROFILING.md)"


def dominant_roofline(table, ms_per_step, tokens, peak, peak_src, traffic_rec):
    """`roofline` of the kernel family with the largest share of the step (pure function of the per-kernel table, so that it is
    tested on the CPU against the committed bench line).  HBM families: algorithmic bytes / CUDA-event time against the measured
    copy bandwidth.  The fused unit-encoder data gradient moves almost no HBM bytes (1 GB per step): its roof is the tensor pipe --
    2 x 3 (3xTF32) x rows x 128 x 128 flops over its time against the measured dense tf32 rate."""
    fam = {}
    for label, (names, _) in KERNEL_FAMILIES.items():
        fam[label] = (sum(table[n]["ms"] for n in names if n in table), sum(table[n]["bytes"] for n in names if n in table))
    dominant = max(fam, key=lambda k: fam[k][0])                        # the family with the largest share of the step
    dom_ms, dom_bytes = fam[dominant]
    traffic = traffic_rec.get(KERNEL_FAMILIES[dominant][1]) if traffic_rec else None
    out = {"kernel": dominant, "traffic": traffic, "algorithmic_bytes_per_step": dom_bytes, "kernel_ms_per_step": dom_ms,
           "share_of_step": dom_ms / ms_per_step if ms_per_step > 0 else 0.0,
           "step_traffic": traffic_rec.get("step_total") if traffic_rec else None}
    hbm_gbs = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    if KERNEL_FAMILIES[dominant][0] == ["unit_dgrad_fused"]:
        tpeak, tsrc = measured_peak_tf32()
        flops = 6.0 * tokens * 40 * 128 * 128                            # 40 unit rows per token, 128 x 128 layer, three tf32 products
        tflops = flops / (dom_ms * 1e-3) / 1e12 if dom_ms > 0 else 0.0
        out.update({"bound": "tensor", "achieved": tflops, "peak": tpeak, "unit": "TFLOP/s", "frac": tflops / tpeak, "peak_source": tsrc,
                    "tensor_flops_per_step": flops, "hbm": {"achieved_GBps": hbm_gbs, "frac": hbm_gbs / peak, "peak": peak},
                    "note": "tensor-pipe work counts the three tf32 products of the 3xTF32 split; the kernel is bound by neither roof but by "
                            "its CUDA-core epilogue and pipeline latency (DESIGN.md 9.1); HBM terms of the same launches under `hbm`"})
    else:
        out.update({"bound": "hbm", "achieved": hbm_gbs, "peak": peak, "unit": "GB/s", "frac": hbm_gbs / peak, "peak_source": peak_src,
                    "note": "bound/frac are HBM terms (algorithmic bytes); the K = 128 layers of the GEMM families also sit at ~0.5 of the "
                            "tf32 tensor peak because every product is three MMAs (3xTF32) -- DESIGN.md 9.1"})
    return out


def recurrence_roofline(cfg, meas, peak):
    """The kernel north_star names: recurrence forward + backward (+ the GAE scan of the prep pass), ALGORITHMIC bytes
    (SURVEY.md 8(d): 12*N*(G+1)*H, + 16*N for GAE) over the CUDA-event time of those launches."""
    k = meas["kernels"]
    rnn_ms = k.get("rnn_fwd", 0.0) + k.get("rnn_bwd", 0.0)
    by = algorithmic_rnn_bytes(cfg)
    n_tok = cfg["batch"] * cfg["seq_len"]
    gae_ms = meas["prep_kernels"].get("gae_scan", 0.0)
    out = {"ms_per_step": rnn_ms, "fwd_ms": k.get("rnn_fwd", 0.0), "bwd_ms": k.get("rnn_bwd", 0.0), "algorithmic_bytes": by,
           "GBps": by / (rnn_ms * 1e-3) / 1e9 if rnn_ms > 0 else 0.0,
           "us_per_sequential_step": 1e3 * rnn_ms / (2 * cfg["seq_len"]) if rnn_ms > 0 else 0.0}
    out["frac"] = out["GBps"] / peak
    out["gae"] = {"ms": gae_ms, "algorithmic_bytes": 16.0 * n_tok, "GBps": 16.0 * n_tok / (gae_ms * 1e-3) / 1e9 if gae_ms > 0 else 0.0,
                  "note": "prep pass (once per iteration, optimizer.py:417-421); 16 B/token is launch-latency bound at this size"}
    tot = rnn_ms + gae_ms
    out["lstm_plus_gae"] = {"ms": tot, "GBps": (by + 16.0 * n_tok) / (tot * 1e-3) / 1e9 if tot > 0 else 0.0}
    out["lstm_plus_gae"]["frac"] = out["lstm_plus_gae"]["GBps"] / peak
    return out


def torch_cuda_baseline(cfg, steps=3, warmup=2):
    """BASELINE.md section 3's "more honest" comparison: the reference's own train() (oracle port, stock torch ops) moved to
    cuda:0 -- cuDNN RNN + cuBLAS + eager autograd, TF32 off so the arithmetic is fp32 like ours.  Reported next to our number;
    like cpu_baseline it only times the oracle, nothing of it is on the product path."""
    import copy
    import torch
    from oracle import ref_optimizer as RO
    from oracle.ref_policy import RefPolicy
    from dotaclient_b200.synthetic import make_rollout
    dev = torch.device("cuda", torch.cuda.current_device())
    S, H, cell, B = cfg["seq_len"], cfg["hidden"], cfg["cell"], cfg["batch"]
    prev = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        torch.manual_seed(7)
        cpu = RO.RefOptimizer(RefPolicy(H, cell), seq_len=S)
        proto = cpu.experiences_from_rollout(make_rollout(S, 7))[0]          # one prepared sequence, replicated B times

        def to_dev(v):
            return v.to(dev) if torch.is_tensor(v) else v
        seqs = []
        for _ in range(B):
            e = copy.copy(proto)
            e.observations = {k: to_dev(v) for k, v in proto.observations.items()}
            e.actions = {k: to_dev(v) for k, v in proto.actions.items()}
            e.masks = {k: to_dev(v) for k, v in proto.masks.items()}
            e.log_probs_sel = {k: to_dev(v) for k, v in proto.log_probs_sel.items()}
            e.hidden = tuple(to_dev(h) for h in proto.hidden) if isinstance(proto.hidden, tuple) else to_dev(proto.hidden)
            e.advantages, e.returns = to_dev(proto.advantages), to_dev(proto.returns)
            seqs.append(e)
        gpu = RO.RefOptimizer(RefPolicy(H, cell).to(dev), seq_len=S)
        for _ in range(warmup):
            gpu.train(seqs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            gpu.train(seqs)
        torch.cuda.synchronize()
        ms = 1e3 * (time.perf_counter() - t0) / steps
        return {"value": 1000.0 / ms, "unit": "steps/s", "ms_per_step": ms, "kind": "oracle port of optimizer.py:581-689 on cuda:0",
                "stack": "stock torch %s eager: cuDNN GRU/LSTM, cuBLAS fp32 (TF32 off), autograd" % torch.__version__,
                "batch": B, "steps": steps}
    except Exception as e:                                                   # e.g. out of memory at a large config
        return {"unavailable": "%s: %s" % (type(e).__name__, str(e)[:200])}
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
        torch.cuda.empty_cache()


def main():
    # stdout carries exactly one JSON line: libraries that chat on fd 1 (NCCL prints its version banner there at the first
    # collective) are sent to stderr for the whole run; emit() writes to the saved descriptor.
    global _REAL_STDOUT
    try:
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        _REAL_STDOUT = saved
    except OSError:                                  # no usable stderr: keep the plain stdout
        _REAL_STDOUT = None
    args = parse_args()
    cfg = resolve_config(args)
    cfg["name"] = args.config
    if cfg.get("stream"):
        run_stream(args, cfg)
        return
    if args.impl == "reference":
        run_reference_arm(args, cfg)
        return
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl")
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus
    dev = torch.device("cuda", local_rank)
    B, S, H, cell = cfg["batch"], cfg["seq_len"], cfg["hidden"], cfg["cell"]
    peak, peak_src = measured_peak_hbm()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    meas = measure_config(cfg, args, world, rank, dev, args.steps, args.warmup, with_e2e=not args.skip_e2e,
                          dump=args.dump_outputs is not None and rank == 0)
    clocks = sampler.stop() if rank == 0 else None

    # the other single-GPU-sized BASELINE configurations (per-GPU shapes of C1 / C3 / C4), 3 timed steps each: driver-timed
    # evidence for every width the kernels serve.  N = 1 runs only (the scaling run times the headline workload).
    extras = {}
    if world == 1 and args.config == "c2" and not args.no_extra and args.batch is None and args.hidden is None and args.seq_len is None:
        for name in ("c1", "c3", "c4"):
            ecfg = dict(CONFIGS[name], name=name)
            try:
                m = measure_config(ecfg, args, world, rank, dev, 3, 3, with_e2e=False)
                rr = recurrence_roofline(ecfg, m, peak)
                extras[name] = {"config": workload_config(ecfg, 1, "hbm"), "ms_per_step": m["ms_per_step"],
                                "global_optimizer_steps_per_sec": 1000.0 / m["ms_per_step"],
                                "env_steps_per_sec": 1000.0 / m["ms_per_step"] * ecfg["batch"] * ecfg["seq_len"],
                                "prep_ms": m["prep_ms"], "gpu_launches_per_step": m["launches"] / 3.0, "cuda_graph": m["cuda_graph"],
                                "ms_per_step_launch_by_launch": m["ms_per_step_launch_by_launch"],
                                "host_enqueue_ms_per_step": m["host_enqueue_ms"], "steps": 3, "warmup": 3,
                                "roofline_recurrence": rr,
                                "top_kernels_ms": dict(sorted(m["kernels"].items(), key=lambda kv: -kv[1])[:6])}
            except Exception as e:                                   # never lose the headline line to an extra
                extras[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:300])}
                torch.cuda.empty_cache()

    if rank != 0:
        finish_process(world)
        return
    ms_per_step = meas["ms_per_step"]
    value = world * 1000.0 / ms_per_step
    tokens = B * S
    # Per-kernel table (CUDA events on the launching stream, averaged per step) with each kernel's ALGORITHMIC HBM bytes
    # (DESIGN.md section 4: inputs read once + outputs written once) -> achieved GB/s and fraction of the measured HBM peak.
    table = kernel_table(meas, peak)
    traffic_rec = None                                                  # measured DRAM bytes per step (ncu), if captured for this shape
    try:
        if (B, S, H) == (CONFIGS[args.config]["batch"], CONFIGS[args.config]["seq_len"], CONFIGS[args.config]["hidden"]):
            with open(os.path.join(ROOT, "profiles", "kernel_traffic.json")) as f:
                traffic_rec = json.load(f).get("%s_%s" % (args.config, cell))
    except Exception:
        pass
    roofline = dominant_roofline(table, ms_per_step, tokens, peak, peak_src, traffic_rec)
    roofline["recurrence"] = recurrence_roofline(cfg, meas, peak)
    roofline["kernels"] = table
    line = {
        "metric": "optimizer_steps_per_sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(cfg, world, "hbm"),
        "value_definition": "n_gpus x (1000 / ms_per_step): per-GPU-batch train() steps per second summed over ranks (weak scaling). "
                            "One data-parallel step is ONE optimizer update on an n_gpus-times larger batch: see "
                            "global_optimizer_steps_per_sec",
        "global_optimizer_steps_per_sec": 1000.0 / ms_per_step, "sequences_per_sec": value * B,
        "env_steps_per_sec": value * tokens,
        "prep": {"ms_per_iteration": meas["prep_ms"], "kernels_ms": meas["prep_kernels"],
                 "what": "experience prep of one iteration's %d rollouts in one batched pass (optimizer.py:328-430): raw rollouts H2D, "
                         "encoder, recurrence, heads, old log-probs, segmented GAE; runs once per iteration, train() `epochs` times" % B,
                 "ms_per_step_prep_plus_train": meas["prep_ms"] + ms_per_step},
        "gpu_launches": meas["launches"], "host_enqueue_ms_per_step": meas["host_enqueue_ms"],
        "launch": {"cuda_graph": meas["cuda_graph"], "kernels_per_step": meas["launches"] / float(args.steps),
                   "ms_per_step_launch_by_launch": meas["ms_per_step_launch_by_launch"],
                   "host_enqueue_ms_per_step_launch_by_launch": meas["host_enqueue_ms_launch_by_launch"],
                   "note": "value/ms_per_step: the step replayed from its CUDA graph (one graph launch per step, same kernels); the "
                           "per-kernel table of `roofline` is measured launch by launch with CUDA events around every call"},
        "roofline": roofline, "clocks": clocks,
    }
    if "ms_e2e" in meas:
        line["e2e"] = {"value": world * 1000.0 / meas["ms_e2e"], "unit": "steps/s", "h2d_bytes_per_step": meas["h2d_bytes"],
                       "d2h_bytes_per_step": 80, "ms_per_step": meas["ms_e2e"],
                       "mode": "double-buffered: DotaOptimizer.prefetch() uploads step k+1 from pinned host memory into the second set of "
                               "graph input buffers while the graph of step k runs",
                       "serial_value": world * 1000.0 / meas["ms_e2e_serial"], "serial_ms_per_step": meas["ms_e2e_serial"]}
        if "ms_e2e_list_api" in meas:
            line["e2e"]["reference_api_value"] = world * 1000.0 / meas["ms_e2e_list_api"]
            line["e2e"]["reference_api_note"] = "train(list of %d device-resident Sequence records): the reference's call signature " \
                                                "(optimizer.py:581), the list is re-stacked on every call like optimizer.py:587-615" % B
    if extras:
        line["extra_configs"] = extras
    if not args.no_cpu_baseline and world == 1:      # reported baselines: rank 0 at N=1 only
        log("timing the stock-torch cuda:0 baseline (oracle port)")
        line["torch_cuda_baseline"] = torch_cuda_baseline(cfg)
        log("timing the CPU baseline (oracle port)")
        v, cores, sample, b_sample = cpu_reference_steps_per_sec(cfg, budget_s=20.0)
        line["cpu_baseline"] = {"value": v, "unit": "steps/s", "cores": cores, "kind": "port", "sample": sample,
                                "sample_batch": b_sample, "scale_factor": b_sample / float(B)}
    if args.dump_outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in meas["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
        log("wrote %d arrays of the last timed step to %s" % (len(meas["outputs"]), args.dump_outputs))
    emit(line)
    finish_process(world)


def finish_process(world):
    """Orderly end of a rank: everything on the device done, all ranks at the barrier, process group destroyed -- under a
    watchdog, so that a teardown problem can never hold the driver's torchrun after the JSON line is out."""
    import torch
    import torch.distributed as dist
    if world <= 1:
        return
    def bail():
        os._exit(0)
    t = threading.Timer(30.0, bail)
    t.daemon = True
    t.start()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    t.cancel()


if __name__ == "__main__":
    main()
