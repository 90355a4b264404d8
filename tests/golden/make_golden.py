"""Generates the fixtures under tests/golden/ by running the REAL reference in place.

Needs a checkout of the reference (``oracle/reference_shim.py``, ``DOTACLIENT_REFERENCE``):
python tests/golden/make_golden.py
The reference (TimZaman/dotaclient @ 8615b90) ships no golden vectors of its own (SURVEY.md 4), so
these fixtures -- outputs of the unmodified reference ``DotaOptimizer.experiences_from_rollout`` and
``DotaOptimizer.train`` (``optimizer.py:328-430,581-689``) on a seeded synthetic rollout -- are what
pins the oracle (``oracle/``) and, through it, the CUDA path.  Nothing is copied from the reference;
only its outputs are recorded.

The weights after training (765 k floats, 3 MB) are stored per tensor as the SHA-256 of their float32
bytes and a fixed seeded sample of SAMPLE elements, which keeps every file far below 1 MB.
"""
import copy
import hashlib
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import reference_shim  # noqa: E402
from dotaclient_b200.synthetic import make_rollout  # noqa: E402

HEADS = ("enum", "x", "y", "target_unit", "ability")
SEQ_LEN, ROLLOUT_LEN, ROLLOUT_SEED, EPOCHS = 16, 40, 11, 3
LOSS_KEYS = ("loss", "policy_loss", "entropy_loss", "value_loss")
SAMPLE = 256
HERE = os.path.dirname(os.path.abspath(__file__))


def record_state_dict(sd, prefix, out):
    """Adds ``<prefix>sha256.<name>``, ``<prefix>idx.<name>`` and ``<prefix>val.<name>`` for every tensor."""
    rng = np.random.RandomState(0)
    for name, t in sd.items():
        flat = t.detach().reshape(-1).numpy()
        idx = np.sort(rng.choice(flat.size, min(flat.size, SAMPLE), replace=False)).astype(np.int64)
        out[prefix + "sha256." + name] = np.array(hashlib.sha256(flat.tobytes()).hexdigest())
        out[prefix + "idx." + name] = idx
        out[prefix + "val." + name] = flat[idx].copy()


def record_ragged_seq8():
    """reference_ragged_seq8.npz: prep of a ragged 29-step rollout (seed 5) into 8-step sequences, then 2 train() epochs."""
    torch.set_num_threads(1)
    ref = reference_shim.make_reference_optimizer(seq_len=8)
    with torch.no_grad():
        xs = ref.experiences_from_rollout(copy.deepcopy(make_rollout(29, 5)))
    out = {"advantages": np.stack([s.advantages.numpy() for s in xs]), "returns": np.stack([s.returns.numpy() for s in xs]),
           "hidden": np.stack([s.hidden.numpy() for s in xs])}
    losses, ents, norms = [], [], []
    for _ in range(2):
        l, e, g = ref.train(xs)
        losses.append(np.stack([l[k].detach().numpy() for k in LOSS_KEYS]))
        ents.append(np.stack([e[k].detach().numpy() for k in HEADS]))
        norms.append(np.stack([g[k].detach().numpy() for k in ("unclipped", "clipped")]))
    out.update(losses=np.stack(losses), entropies=np.stack(ents), grad_norms=np.stack(norms))
    record_state_dict(ref.policy_base.state_dict(), "final_", out)
    path = os.path.join(HERE, "reference_ragged_seq8.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def _reference_rank_worker(rank, world, port, out_dir):
    """Runs the UNMODIFIED reference distributed.py + optimizer.train under gloo (SURVEY.md 0.4: prep through policy_base)."""
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    O, P, D = reference_shim.load()
    opt = reference_shim.make_reference_optimizer(seq_len=8)
    with torch.no_grad():
        xs = opt.experiences_from_rollout(make_rollout(24, 300 + rank))
    opt.policy = D.DistributedDataParallelSparseParamCPU(opt.policy_base)
    opt.optimizer = torch.optim.Adam(opt.policy.parameters(), lr=5e-5)
    recs = []
    for _ in range(2):
        l, e, g = opt.train(xs)
        recs.append(([float(l[k]) for k in LOSS_KEYS], float(g["unclipped"]), float(g["clipped"])))
    torch.save({"recs": recs, "sd": opt.policy_base.state_dict()}, os.path.join(out_dir, "ref_rank%d.pt" % rank))
    dist.destroy_process_group()


def record_gloo_world2():
    """reference_gloo_world2.npz: two gloo ranks (rollouts of 24 steps, seeds 300 + rank) through the reference's
    DistributedDataParallelSparseParamCPU, 2 train() epochs; per rank the losses, grad norms and final weights."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_reference_rank_worker, args=(2, port, tmp), nprocs=2, join=True)
        for r in range(2):
            rec = torch.load(os.path.join(tmp, "ref_rank%d.pt" % r))
            out["rank%d_losses" % r] = np.array([ep[0] for ep in rec["recs"]], dtype=np.float64)
            out["rank%d_grad_norms" % r] = np.array([[ep[1], ep[2]] for ep in rec["recs"]], dtype=np.float64)
            record_state_dict(rec["sd"], "rank%d_final_" % r, out)
    path = os.path.join(HERE, "reference_gloo_world2.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def main():
    torch.set_num_threads(1)          # bit-stable reductions
    ref = reference_shim.make_reference_optimizer(seq_len=SEQ_LEN)
    init_sums = {k: float(v.double().sum()) for k, v in ref.policy_base.state_dict().items()}
    data = make_rollout(ROLLOUT_LEN, ROLLOUT_SEED)
    with torch.no_grad():
        seqs = ref.experiences_from_rollout(copy.deepcopy(data))
    out = {"seq_len": SEQ_LEN, "rollout_len": ROLLOUT_LEN, "rollout_seed": ROLLOUT_SEED, "epochs": EPOCHS}
    out["advantages"] = np.stack([s.advantages.numpy() for s in seqs])
    out["returns"] = np.stack([s.returns.numpy() for s in seqs])
    out["values"] = np.stack([s.values.numpy().reshape(-1) for s in seqs])
    out["hidden"] = np.stack([s.hidden.numpy().reshape(-1) for s in seqs])
    for k in HEADS:
        out["old_logp_" + k] = torch.cat([s.log_probs_sel[k] for s in seqs]).numpy()
    # forward at the initial weights on the stacked batch (what train() sees at :619)
    obs = {k: torch.stack([s.observations[k] for s in seqs]) for k in ref.policy_base.INPUT_KEYS}
    hidden = torch.cat([s.hidden for s in seqs], dim=1)
    with torch.no_grad():
        logits, values, _ = ref.policy_base(**obs, hidden=hidden)
    for k in HEADS:
        out["logits_" + k] = logits[k].numpy()
    out["forward_values"] = values.numpy()
    losses, ents, gns = [], [], []
    for ep in range(EPOCHS):
        l, e, g = ref.train(seqs)
        losses.append([float(l[k]) for k in ("loss", "policy_loss", "entropy_loss", "value_loss")])
        ents.append([float(e[k]) for k in HEADS])
        gns.append([float(g["unclipped"]), float(g["clipped"])])
        if ep == 0:
            names = [n for n, _ in ref.policy_base.named_parameters()]
            out["param_names"] = np.array(names)
            out["grad_norms_ep0"] = np.array([float(p.grad.norm(2)) if p.grad is not None else -1.0
                                              for _, p in ref.policy_base.named_parameters()])
            out["grad_rnn_bias_hh_ep0"] = dict(ref.policy_base.named_parameters())["rnn.bias_hh_l0"].grad.numpy().copy()
            out["grad_value_w_ep0"] = dict(ref.policy_base.named_parameters())["affine_value.weight"].grad.numpy().copy()
    out["losses"] = np.array(losses, dtype=np.float64)
    out["entropies"] = np.array(ents, dtype=np.float64)
    out["grad_norms"] = np.array(gns, dtype=np.float64)
    sd = ref.policy_base.state_dict()
    out["init_param_sums"] = np.array([init_sums[k] for k in sd])
    out["final_param_sums"] = np.array([float(v.double().sum()) for v in sd.values()])
    out["final_param_abs_sums"] = np.array([float(v.double().abs().sum()) for v in sd.values()])
    out["final_rnn_bias_hh"] = sd["rnn.bias_hh_l0"].numpy().copy()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_h256_gru.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")
    # GAE known-answer vector (SURVEY.md 4), from the reference's advantage_returns itself
    O, _, _ = reference_shim.load()
    r = np.array([1, 1, 1, 0], np.float32)
    v = np.array([.5, .5, .5, 0], np.float32)
    a, q = O.advantage_returns(r, v, 0.98, 0.97)
    rng = np.random.RandomState(3)
    r2 = np.append(rng.randn(300).astype(np.float32), np.float32(0))
    v2 = np.append(rng.randn(300).astype(np.float32), np.float32(0))
    a2, q2 = O.advantage_returns(r2, v2, 0.98, 0.97)
    np.savez_compressed(os.path.join(os.path.dirname(path), "gae_reference.npz"), r=r, v=v, adv=a, ret=q, r2=r2, v2=v2,
                        adv2=a2, ret2=q2)
    record_ragged_seq8()
    record_gloo_world2()


if __name__ == "__main__":
    main()
