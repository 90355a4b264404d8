"""CPU tests of the host-side logic: flat parameter space, the DDP wrapper over gloo (world_size 2),
the in-process MessageQueue, Sequence records, CLI flags, the synthetic generator."""
import os
import pickle
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dotaclient_b200.flat import FlatParameterSpace, head_dependency
from dotaclient_b200.synthetic import HEAD_SIZES, OBS_SHAPES, make_rollout, ragged_lengths


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


# ------------------------------------------------------------------------------------------------ policy surface
def test_policy_state_dict_matches_reference_layout():
    """34 keys in the reference's order and shapes (SURVEY.md 2.2), identical seeded init to the oracle restatement."""
    from dotaclient_b200.policy import Policy
    from oracle.ref_policy import RefPolicy
    for H, cell in ((256, "gru"), (128, "lstm")):
        torch.manual_seed(7)
        mine = Policy(hidden_size=H, cell=cell)
        torch.manual_seed(7)
        ref = RefPolicy(H, cell)
        a, b = mine.state_dict(), ref.state_dict()
        assert list(a.keys()) == list(b.keys()) and len(a) == 34
        for k in a:
            assert a[k].shape == b[k].shape and torch.equal(a[k], b[k]), k
    assert Policy().hidden_size == 256 and Policy().cell == "gru"
    assert Policy.MAX_UNITS == 40 and list(Policy.OUTPUT_KEYS) == ["enum", "x", "y", "target_unit", "ability"]
    assert Policy().init_hidden().shape == (1, 1, 256)


def test_policy_rejects_cpu_inputs():
    from dotaclient_b200.policy import Policy
    pol = Policy(hidden_size=128, cell="gru")
    r = make_rollout(4, 1)
    with pytest.raises(RuntimeError, match="CUDA only"):
        pol.sequence(hidden=pol.init_hidden(), **r["observations"])


def test_policy_class_helpers():
    from dotaclient_b200.policy import Policy
    sel = Policy.flatten_selections({"enum": 1, "x": 3, "y": 8})
    assert sel["x"].tolist().index(True) == 3 and not sel["ability"].any() and sel["target_unit"].shape == (40,)
    hm = Policy.head_masks({"enum": 0, "ability": 2})
    assert hm["enum"].all() and hm["ability"].all() and not hm["x"].any() and hm["x"].shape == (1, 1, 9)
    lp = Policy.masked_softmax(torch.tensor([[[0.0, 1.0, 2.0]]]), torch.tensor([[[True, True, False]]]))
    assert torch.allclose(lp[0, 0, :2].exp().sum(), torch.tensor(1.0))

    class Ability:
        def __init__(self, slot, ok):
            self.slot, self.is_activated, self.level, self.cooldown_remaining, self.is_fully_castable = slot, ok, 1, 0, ok

    class Unit:
        is_alive = True
        abilities = [Ability(0, False), Ability(1, False), Ability(2, False), Ability(5, True)]
    handles = np.full(40, -1)
    m = Policy.action_masks(Unit(), handles)
    assert not m["ability"].any() and not m["enum"][0, 0, 3] and not m["enum"][0, 0, 2] and m["enum"][0, 0, 1]
    handles[[0, 7]] = 5
    m = Policy.action_masks(Unit(), handles)
    assert m["target_unit"][0, 0].nonzero().flatten().tolist() == [7] and m["enum"][0, 0, 2]
    Unit.is_alive = False
    m = Policy.action_masks(Unit(), handles)
    assert m["enum"][0, 0].tolist() == [True, False, False, False] and not m["x"].any()


# ------------------------------------------------------------------------------------------------ flat space
def test_flat_parameter_space_views_and_state_dict():
    from dotaclient_b200.policy import Policy
    torch.manual_seed(7)
    pol = Policy(hidden_size=128, cell="lstm")
    before = {k: v.clone() for k, v in pol.state_dict().items()}
    flat = FlatParameterSpace(pol)
    assert flat.n_seg == 34 and flat.total >= sum(v.numel() for v in before.values())
    assert all(lo % 64 == 0 for lo in flat.starts) and flat.ends[-1] <= flat.total
    assert flat.names == list(before.keys())
    for k, v in pol.state_dict().items():
        assert torch.equal(v, before[k])
    # parameters and gradients are views into the flat buffers
    flat.param.zero_()
    assert all(float(p.abs().sum()) == 0 for p in pol.parameters())
    pol.load_state_dict(before)
    assert torch.equal(flat.param[:before["affine_env.weight"].numel()], before["affine_env.weight"].flatten())
    p = pol.affine_value.weight
    p.grad.fill_(2.0)
    assert float(flat.grad_of("affine_value.weight").sum()) == 2.0 * p.numel()
    flat.zero_grad()
    assert float(flat.grad_full.abs().sum()) == 0.0 and p.grad.data_ptr() == flat.grad_of("affine_value.weight").data_ptr()
    # which parameters only get a gradient through a particular head (optimizer.py:627-630, policy.py:127)
    dep = dict(zip(flat.names, flat.seg_head.tolist()))
    assert dep["affine_unit_attention.weight"] == 3 and dep["affine_unit_eth.bias"] == 3
    assert dep["affine_head_enum.weight"] == 0 and dep["affine_move_y.bias"] == 2 and dep["affine_head_ability.bias"] == 4
    assert dep["affine_value.weight"] == 5 and dep["rnn.weight_hh_l0"] == -1 and dep["affine_unit_enh.weight"] == -1
    assert head_dependency("affine_pre_rnn.bias") == -1


def test_autograd_accumulates_into_flat_views():
    m = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 1))
    flat = FlatParameterSpace(m)
    flat.zero_grad()
    m(torch.ones(2, 4)).sum().backward()
    for p, lo, hi in zip(m.parameters(), flat.starts, flat.ends):
        assert torch.equal(p.grad.flatten(), flat.grad[lo:hi])
    assert float(flat.grad.abs().sum()) > 0
    for p, lo in zip(m.parameters(), flat.offsets):
        assert p.grad.data_ptr() == flat.grad[lo:].data_ptr()


def test_detached_grads_gathered_into_flat_buffer():
    """train()'s gradient path: .grad detached before backward (autograd hands tensors over without an accumulate kernel per
    parameter), then one multi-tensor copy into the flat buffer; parameters without a gradient stay zero and every .grad
    is a flat view again afterwards."""
    m = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 1), torch.nn.Linear(2, 2))     # the last layer is unused
    twin = torch.nn.Sequential(torch.nn.Linear(4, 3), torch.nn.Linear(3, 1), torch.nn.Linear(2, 2))
    twin.load_state_dict(m.state_dict())
    flat = FlatParameterSpace(m)
    flat.grad.fill_(7.0)                                       # stale contents must not survive
    flat.zero_grad_detached()
    assert all(p.grad is None for p in m.parameters()) and float(flat.grad_full.abs().sum()) == 0.0
    x = torch.arange(8.0).reshape(2, 4)
    m[1](m[0](x)).sum().backward()
    twin[1](twin[0](x)).sum().backward()
    assert m[0].weight.grad.data_ptr() != flat.grad_of("0.weight").data_ptr()      # handed over, not accumulated in place
    flat.gather_grads()
    for (name, p), q in zip(m.named_parameters(), twin.parameters()):
        assert p.grad.data_ptr() == flat.grad_of(name).data_ptr()
        expect = q.grad if q.grad is not None else torch.zeros_like(q)
        assert torch.equal(p.grad, expect), name
    flat.gather_grads()                                        # idempotent when the views are already attached
    assert torch.equal(m[0].weight.grad, twin[0].weight.grad)


# ------------------------------------------------------------------------------------------------ DDP over gloo
def _ddp_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from dotaclient_b200.distributed import DistributedDataParallelSparseParamCPU
    torch.manual_seed(100 + rank)                       # ranks start from DIFFERENT weights
    net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 2))
    ddp = DistributedDataParallelSparseParamCPU(net)
    synced = ddp.flat.param.clone()
    torch.manual_seed(7 + rank)
    x = torch.randn(8, 6)
    ddp.flat.zero_grad()
    ddp(x).pow(2).sum().backward()                      # hook -> ONE all-reduce + count-divide
    hooked = ddp.flat.grad.clone()
    # sparse case: rank 1 has no gradient for the last layer -> average over the ranks that do (distributed.py:36-57)
    ddp.flat.zero_grad()
    ddp.auto_reduce = False
    ddp(x).pow(2).sum().backward()
    local = ddp.flat.grad.clone()
    has = [1.0] * ddp.flat.n_seg
    if rank == 1:
        lo = ddp.flat.offsets[2]
        ddp.flat.grad[lo:].zero_()
        local[lo:] = 0
        has[2] = has[3] = 0.0
    ddp.set_local_flags(has)
    ddp.allreduce_gradients(divide=True, flags_ready=True)
    def compact(v):          # drop the alignment padding between tensors
        return torch.cat([v[a:b] for a, b in zip(ddp.flat.starts, ddp.flat.ends)])
    torch.save({"synced": compact(synced), "hooked": compact(hooked), "local": compact(local),
                "sparse": compact(ddp.flat.grad.clone()), "counts": ddp.flat.flags.clone(), "x": x},
               os.path.join(out_dir, "r%d.pt" % rank))
    dist.destroy_process_group()


def test_ddp_wrapper_gloo_world2(tmp_path):
    port = _free_port()
    mp.spawn(_ddp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    assert torch.equal(r0["synced"], r1["synced"])                       # broadcast from rank 0 (distributed.py:71-74)
    torch.manual_seed(100)
    ref = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 2))
    assert torch.equal(r0["synced"], torch.cat([p.detach().flatten() for p in ref.parameters()]))
    # dense case == mean of the two ranks' local gradients, identical on both ranks
    grads = []
    for r in (r0, r1):
        ref.zero_grad()
        ref(r["x"]).pow(2).sum().backward()
        grads.append(torch.cat([p.grad.flatten() for p in ref.parameters()]))
    torch.testing.assert_close(r0["hooked"], (grads[0] + grads[1]) / 2)
    assert torch.equal(r0["hooked"], r1["hooked"])
    # sparse case: counts [2,2,1,1]; last layer == rank 0's gradient alone, applied on BOTH ranks (documented fix)
    assert r0["counts"].tolist() == [2.0, 2.0, 1.0, 1.0]
    lo = 6 * 5 + 5
    torch.testing.assert_close(r0["sparse"][:lo], (grads[0][:lo] + grads[1][:lo]) / 2)
    torch.testing.assert_close(r0["sparse"][lo:], grads[0][lo:])
    assert torch.equal(r0["sparse"], r1["sparse"])


def test_ddp_wrapper_forwards_module_api():
    """init_hidden / sequence / single are reachable through the wrapper (the reference's wrapper lacks them)."""
    from dotaclient_b200.distributed import DistributedDataParallelSparseParamCPU
    from dotaclient_b200.policy import Policy
    pol = Policy(hidden_size=128, cell="gru")
    ddp = DistributedDataParallelSparseParamCPU(pol)
    assert ddp.init_hidden().shape == (1, 1, 128) and ddp.module is pol
    assert [k for k, _ in ddp.named_parameters()][0] == "module.affine_env.weight"


# ------------------------------------------------------------------------------------------------ broker + records
def test_message_queue_in_process_roundtrip():
    from dotaclient_b200.optimizer import MessageQueue
    a = MessageQueue(host="h", port=1, prefetch_count=1, use_model_exchange=True)
    b = MessageQueue(host="h", port=1, prefetch_count=1, use_model_exchange=False)
    a.connect(), b.connect()
    assert a.xp_queue_size == 0 and a.latest_model() is None
    body = pickle.dumps(make_rollout(5, 3, with_canvas=True))
    b.publish_experience(body)
    assert a.xp_queue_size == 1
    method, props, got = a.consume_xp()
    assert got == body and method.delivery_tag == 1 and a.xp_queue_size == 0
    a.publish_model(b"weights", {"version": 4})
    a.publish_model(b"weights2", {"version": 5})                       # recent-history length 1: last one wins
    assert b.latest_model() == (b"weights2", {"version": 5})
    a.process_data_events()
    a.close()


def test_sequence_lazy_compact_logprobs_and_dense_roundtrip():
    from dotaclient_b200.optimizer import Sequence
    r = make_rollout(12, 4)
    dense = torch.randn(12, 5)
    s = Sequence(0, 1, 2, r["observations"], r["actions"], r["masks"], torch.zeros(1, 12, 1), r["rewards"],
                 torch.zeros(1, 1, 8), old_logp=dense)
    lp = s.log_probs_sel
    for h, k in enumerate(("enum", "x", "y", "target_unit", "ability")):
        step = r["actions"][k].any(dim=1)
        assert torch.equal(lp[k], dense[step, h]) and lp[k].numel() == int(step.sum())
    s2 = Sequence(0, 1, 2, r["observations"], r["actions"], r["masks"], None, None, None, log_probs_sel=lp)
    d2 = s2.dense_old_logp()
    for h, k in enumerate(("enum", "x", "y", "target_unit", "ability")):
        step = r["actions"][k].any(dim=1)
        assert torch.equal(d2[step, h], dense[step, h]) and float(d2[~step, h].abs().sum()) == 0


def test_cli_flags_match_reference_defaults():
    from dotaclient_b200.optimizer import build_arg_parser
    a = build_arg_parser().parse_args([])
    assert (a.epochs, a.min_seq_per_epoch, a.seq_len, a.learning_rate, a.entropy_coef, a.vf_coef,
            a.mq_prefetch_count, a.ip, a.port) == (4, 1024, 16, 5e-5, 5e-4, 0.5, 1, "127.0.0.1", 5672)
    assert a.hidden_size == 256 and a.cell == "gru"


def test_optimizer_requires_cuda_loudly():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from dotaclient_b200.optimizer import advantage_returns
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        advantage_returns(np.zeros(3, np.float32), np.zeros(3, np.float32), 0.98, 0.97)


# ------------------------------------------------------------------------------------------------ synthetic data
def test_synthetic_rollout_schema_and_determinism():
    r = make_rollout(50, 9)
    r2 = make_rollout(50, 9)
    for k, shp in OBS_SHAPES.items():
        assert r["observations"][k].shape == (50,) + shp and torch.equal(r["observations"][k], r2["observations"][k])
    assert r["rewards"].shape == (50, 10) and r["rewards"].dtype == np.float32
    enum = r["actions"]["enum"].float().argmax(1)
    for k, n in HEAD_SIZES.items():
        a, m = r["actions"][k], r["masks"][k]
        assert a.shape == (50, n) and a.dtype == torch.bool and m.dtype == torch.bool
        assert (a.sum(1) <= 1).all() and (a & ~m).sum() == 0          # one-hot inside the mask
    assert (r["actions"]["x"].any(1) == (enum == 1)).all() and (r["actions"]["y"].any(1) == (enum == 1)).all()
    assert (r["actions"]["target_unit"].any(1) == (enum == 2)).all() and (r["actions"]["ability"].any(1) == (enum == 3)).all()
    assert not r["masks"]["target_unit"][:, 0].any()
    assert all(8 <= L <= 48 for L in ragged_lengths(20, 16, 0))


# ------------------------------------------------------------------------------------------------ bench / tools host logic
def test_bench_config_is_identical_in_both_arms_and_names_the_workload():
    """The driver compares the `config` of `bench.py` and `bench.py --impl reference`: both come from workload_config()."""
    import bench
    cfg = dict(bench.CONFIGS["c2"])
    a = bench.workload_config(cfg, 1, "hbm")
    b = bench.workload_config(cfg, 1, "cpu")
    assert a == b and a["batch_per_gpu"] == 256 and a["seq_len"] == 512 and a["hidden"] == 128 and "workload" in a
    assert bench.workload_config(cfg, 8, "hbm")["global_batch"] == 2048
    assert bench.algorithmic_rnn_bytes(cfg) == 12.0 * 256 * 512 * 5 * 128            # SURVEY.md 8(d), LSTM: G + 1 = 5


def test_bench_step_outputs_names_dtypes_and_sampling():
    """--dump-outputs: one float array per returned scalar and per parameter, a wide cell's recurrent weights sampled at the
    same positions on every call, the whole dump under 64 MB even at the widest cell the recurrence accepts (H = 2048)."""
    import types
    import bench
    from dotaclient_b200.policy import Policy
    keys = ("enum", "x", "y", "target_unit", "ability")
    result = ({k: torch.tensor(float(i)) for i, k in enumerate(("loss", "policy_loss", "entropy_loss", "value_loss"))},
              {k: torch.tensor(0.5) for k in keys}, {"unclipped": torch.tensor(2.0), "clipped": torch.tensor(1.0)})
    torch.manual_seed(7)
    small = types.SimpleNamespace(policy_base=Policy(hidden_size=128, cell="lstm"))
    out = bench.step_outputs(small, result)
    assert len(out) == 4 + 5 + 2 + 34 and float(out["value_loss"]) == 3.0 and float(out["grad_norm.clipped"]) == 1.0
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    for k, v in small.policy_base.state_dict().items():
        assert np.array_equal(out["param." + k], v.numpy()), k                      # BASELINE widths: every element
    wide = types.SimpleNamespace(policy_base=Policy(hidden_size=2048, cell="lstm"))
    a, b = bench.step_outputs(wide, result), bench.step_outputs(wide, result)
    w = wide.policy_base.rnn.weight_hh_l0.detach().reshape(-1).numpy()
    idx = np.sort(np.random.default_rng(0).choice(w.size, bench.DUMP_MAX_ELEMENTS, replace=False))        # the documented positions
    assert np.array_equal(a["param.rnn.weight_hh_l0"], w[idx])
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.nbytes for v in a.values()) <= 64 << 20


def test_kernel_traffic_json_matches_the_committed_ncu_csv(tmp_path):
    """profiles/kernel_traffic.json (read by bench.py for roofline.traffic) is derived from profiles/r2_ncu_traffic_c2.csv."""
    import csv
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    rec = json.load(open(os.path.join(root, "profiles", "kernel_traffic.json")))["c2_lstm"]
    total = 0.0
    for r in csv.reader(open(os.path.join(root, "profiles", "r2_ncu_traffic_c2.csv"))):
        if len(r) >= 15 and r[0].isdigit() and r[12].startswith("dram__bytes"):
            total += float(r[14].replace(",", "")) * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[r[13]]
    assert abs(total - rec["step_total"]) <= 1e-6 * total
    assert 15e9 < rec["step_total"] < 25e9 and rec["gemm_fwd_dgrad"] > rec["rnn"] > 1e9     # 35.2 GB before the fused encoder backward
    assert rec["unit_dgrad_fused"] < 2e9                                                     # ... whose data-gradient kernel moves ~1 GB


def test_dominant_roofline_of_the_committed_bench_line():
    """bench.py's `roofline` names the kernel family with the largest share of the step; checked on the per-kernel table of the
    committed C2 line (profiles/r2_bench_c2_n1.json): the fused unit-encoder data gradient, bound by the tensor pipe, with
    its measured DRAM traffic from profiles/kernel_traffic.json; without it the forward/dgrad GEMM family in HBM terms."""
    import json
    import bench
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    line = json.loads(open(os.path.join(root, "profiles", "r2_bench_c2_n1.json")).read().strip().splitlines()[-1])
    rec = json.load(open(os.path.join(root, "profiles", "kernel_traffic.json")))["c2_lstm"]
    table = line["roofline"]["kernels"]
    r = bench.dominant_roofline(table, line["ms_per_step"], 256 * 512, 6576.7, "measured", rec)
    assert "dc_unit_dgrad_fused" in r["kernel"] and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
    assert abs(r["kernel_ms_per_step"] - table["unit_dgrad_fused"]["ms"]) < 1e-9 and 0.2 < r["share_of_step"] < 0.3
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12 and 0.1 < r["frac"] < 0.6
    assert r["traffic"] == rec["unit_dgrad_fused"] and r["step_traffic"] == rec["step_total"]
    rest = {k: v for k, v in table.items() if k != "unit_dgrad_fused"}
    r2 = bench.dominant_roofline(rest, line["ms_per_step"], 256 * 512, 6576.7, "measured", None)
    assert "dc_gemm_tf32x3" in r2["kernel"] and r2["bound"] == "hbm" and r2["unit"] == "GB/s" and r2["traffic"] is None
    want = (table["gemm_tf32x3"]["bytes"] + table["gemm_unit_max"]["bytes"]) / ((table["gemm_tf32x3"]["ms"] + table["gemm_unit_max"]["ms"]) * 1e-3) / 1e9
    assert abs(r2["achieved"] - want) < 1e-6 * want and abs(r2["frac"] - want / 6576.7) < 1e-9


def test_committed_bench_lines_carry_the_contract_keys():
    """The bench lines kept as evidence under profiles/ (one GPU, 2 / 4 / 8 GPUs, reference arm) have every key of the bench.py
    contract, name the BASELINE metric, and their derived fields are consistent with each other."""
    import json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    base = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
            "data", "config"}
    for name, n in (("r2_bench_c2_n1.json", 1), ("r2_bench_c2_n2.json", 2), ("r2_bench_c2_n4.json", 4), ("r2_bench_c4_n8.json", 8)):
        line = json.loads(open(os.path.join(root, "profiles", name)).read().strip().splitlines()[-1])
        assert base | {"roofline", "gpu_launches", "clocks"} <= set(line), (name, base - set(line))
        assert line["metric"] == "optimizer_steps_per_sec" and line["unit"] == "steps/s" and line["higher_is_better"] is True
        assert line["n_gpus"] == n and line["scaling"] == "weak" and line["dtype"] == "f32" and line["vs_baseline"] is None
        assert abs(line["value"] - n * 1000.0 / line["ms_per_step"]) <= 1e-6 * line["value"]
        assert "workload" in line["config"] and "model" not in line["config"]
        r = line["roofline"]
        assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
        if "c2" in name:                              # the C4 evidence run skipped the end-to-end leg (--skip-e2e)
            assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"]) and line["e2e"]["h2d_bytes_per_step"] > 0
        assert line["gpu_launches"] > 0 and not set(line["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if n == 1:
            cb = line["cpu_baseline"]
            assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] == "port" and cb["value"] > 0
            assert set(line["extra_configs"]) == {"c1", "c3", "c4"} and all("ms_per_step" in v for v in line["extra_configs"].values())
    ref = json.loads(open(os.path.join(root, "profiles", "r2_bench_reference_arm_n1.json")).read().strip().splitlines()[-1])
    assert ref["impl"] == "reference" and base <= set(ref) and ref["metric"] == "optimizer_steps_per_sec"
    assert ref["e2e"]["h2d_bytes_per_step"] == 0 and ref["e2e"]["d2h_bytes_per_step"] == 0 and ref["cpu_baseline"]["value"] == ref["value"]
