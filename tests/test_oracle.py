"""CPU tests: the oracle against the reference's recorded outputs (tests/golden, written by tests/golden/make_golden.py)."""
import copy
import ctypes
import hashlib
import os
import subprocess

import numpy as np
import torch

from oracle import ref_optimizer as RO
from oracle.ref_policy import RefPolicy, masked_softmax, sample_index
from dotaclient_b200.synthetic import make_rollout

HEADS = ("enum", "x", "y", "target_unit", "ability")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _c_gae():
    so = os.path.join(ROOT, "oracle", "libgae_ref.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
    lib = ctypes.CDLL(so)
    lib.gae_ref.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_double, ctypes.c_double,
                            ctypes.c_void_p, ctypes.c_void_p]

    def run(r, v, gamma=0.98, lam=0.97):
        n = len(r) - 1
        a, q = np.empty(n, np.float32), np.empty(n, np.float32)
        lib.gae_ref(r.ctypes.data, v.ctypes.data, n, gamma, lam, a.ctypes.data, q.ctypes.data)
        return a, q
    return run


def test_gae_known_answer(gae_golden):
    """SURVEY.md 4 known-answer vector + a 300-step vector recorded from the reference's advantage_returns."""
    a, q = RO.advantage_returns(gae_golden["r"], gae_golden["v"])
    np.testing.assert_array_equal(a, gae_golden["adv"])
    np.testing.assert_array_equal(q, gae_golden["ret"])
    np.testing.assert_allclose(a, [2.3829143, 1.4653, 0.5], rtol=1e-6)
    np.testing.assert_allclose(q, [2.9404, 1.98, 1.0], rtol=1e-6)
    a2, q2 = RO.advantage_returns(gae_golden["r2"], gae_golden["v2"])
    np.testing.assert_array_equal(a2, gae_golden["adv2"])
    np.testing.assert_array_equal(q2, gae_golden["ret2"])


def test_c_gae_matches_scipy_restatement(gae_golden):
    run = _c_gae()
    a, q = run(gae_golden["r2"], gae_golden["v2"])
    np.testing.assert_array_equal(a, gae_golden["adv2"])
    np.testing.assert_array_equal(q, gae_golden["ret2"])
    rng = np.random.RandomState(0)
    for n in (1, 2, 31, 32, 33, 1000):
        r = np.append(rng.randn(n).astype(np.float32), np.float32(0))
        v = np.append(rng.randn(n).astype(np.float32), np.float32(0))
        a, q = run(r, v)
        a2, q2 = RO.advantage_returns(r, v)
        np.testing.assert_array_equal(a, a2)
        np.testing.assert_array_equal(q, q2)


def test_numpy_reward_sum_order():
    """The GAE kernel reproduces numpy's pairwise add-reduce order for 10 sub-rewards (optimizer.py:397)."""
    rng = np.random.RandomState(1)
    x = (rng.randn(257, 10) * 3).astype(np.float32)
    f = np.float32
    manual = np.array([f(f(f(f(f(r[0] + r[1]) + f(r[2] + r[3])) + f(f(r[4] + r[5]) + f(r[6] + r[7]))) + r[8]) + r[9])
                       for r in x], dtype=np.float32)
    np.testing.assert_array_equal(np.sum(x, axis=1), manual)


def _oracle(seq_len=16):
    torch.manual_seed(7)
    return RO.RefOptimizer(RefPolicy(256, "gru"), seq_len=seq_len)


def test_oracle_reproduces_reference_golden(golden):
    """Oracle == recorded reference outputs, bit for bit (init, prep, forward, three train epochs)."""
    torch.set_num_threads(1)
    opt = _oracle(int(golden["seq_len"]))
    sd = opt.policy_base.state_dict()
    assert list(sd.keys()) == [str(n) for n in golden["param_names"]]
    np.testing.assert_array_equal(np.array([float(v.double().sum()) for v in sd.values()]), golden["init_param_sums"])
    data = make_rollout(int(golden["rollout_len"]), int(golden["rollout_seed"]))
    seqs = opt.experiences_from_rollout(copy.deepcopy(data))
    np.testing.assert_array_equal(np.stack([s.advantages.numpy() for s in seqs]), golden["advantages"])
    np.testing.assert_array_equal(np.stack([s.returns.numpy() for s in seqs]), golden["returns"])
    np.testing.assert_array_equal(np.stack([s.values.numpy().reshape(-1) for s in seqs]), golden["values"])
    np.testing.assert_array_equal(np.stack([s.hidden.numpy().reshape(-1) for s in seqs]), golden["hidden"])
    for k in HEADS:
        np.testing.assert_array_equal(torch.cat([s.log_probs_sel[k] for s in seqs]).numpy(), golden["old_logp_" + k])
    (_, _, _, _, _), logits, values = opt.loss_only(seqs)
    for k in HEADS:
        np.testing.assert_array_equal(logits[k].detach().numpy(), golden["logits_" + k])
    np.testing.assert_array_equal(values.detach().numpy(), golden["forward_values"])
    for ep in range(int(golden["epochs"])):
        l, e, g = opt.train(seqs)
        got = [float(l[k]) for k in ("loss", "policy_loss", "entropy_loss", "value_loss")]
        np.testing.assert_array_equal(np.array(got), golden["losses"][ep])
        np.testing.assert_array_equal(np.array([float(e[k]) for k in HEADS]), golden["entropies"][ep])
        np.testing.assert_array_equal(np.array([float(g["unclipped"]), float(g["clipped"])]), golden["grad_norms"][ep])
    sd = opt.policy_base.state_dict()
    np.testing.assert_array_equal(np.array([float(v.double().sum()) for v in sd.values()]), golden["final_param_sums"])
    np.testing.assert_array_equal(sd["rnn.bias_hh_l0"].numpy(), golden["final_rnn_bias_hh"])


def _load_golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


def _assert_state_dict_matches(sd, golden, prefix):
    """Bit for bit against a state dict recorded by make_golden.record_state_dict: the sampled elements first (a mismatch
    shows its size), then the SHA-256 of every whole tensor."""
    assert sorted(sd) == sorted(k[len(prefix) + 4:] for k in golden.files if k.startswith(prefix + "val."))
    for name, t in sd.items():
        flat = t.detach().reshape(-1).numpy()
        np.testing.assert_array_equal(flat[golden[prefix + "idx." + name]], golden[prefix + "val." + name], err_msg=name)
        assert hashlib.sha256(flat.tobytes()).hexdigest() == str(golden[prefix + "sha256." + name]), name


def test_oracle_bit_identical_to_reference_live():
    """Restatement vs the reference's own run (recorded in tests/golden/reference_ragged_seq8.npz), ragged rollout, 2 epochs."""
    golden = _load_golden("reference_ragged_seq8.npz")
    torch.set_num_threads(1)
    mine = _oracle(8)
    xm = mine.experiences_from_rollout(copy.deepcopy(make_rollout(29, 5)))
    assert len(xm) == len(golden["advantages"]) == 4
    np.testing.assert_array_equal(np.stack([s.advantages.numpy() for s in xm]), golden["advantages"])
    np.testing.assert_array_equal(np.stack([s.returns.numpy() for s in xm]), golden["returns"])
    np.testing.assert_array_equal(np.stack([s.hidden.numpy() for s in xm]), golden["hidden"])
    for ep in range(2):
        lm_, em_, gm_ = mine.train(xm)
        np.testing.assert_array_equal(np.stack([lm_[k].detach().numpy() for k in ("loss", "policy_loss", "entropy_loss",
                                                                                   "value_loss")]), golden["losses"][ep])
        np.testing.assert_array_equal(np.stack([em_[k].detach().numpy() for k in HEADS]), golden["entropies"][ep])
        np.testing.assert_array_equal(np.stack([gm_[k].detach().numpy() for k in ("unclipped", "clipped")]), golden["grad_norms"][ep])
    _assert_state_dict_matches(mine.policy_base.state_dict(), golden, "final_")


def test_oracle_lstm_and_width_variants_run():
    """The widths/cell the reference cannot express: shapes, finite losses, state_dict layout."""
    for H, cell in ((128, "lstm"), (128, "gru"), (512, "lstm")):
        torch.manual_seed(7)
        opt = RO.RefOptimizer(RefPolicy(H, cell), seq_len=8)
        G = 4 if cell == "lstm" else 3
        sd = opt.policy_base.state_dict()
        assert len(sd) == 34 and sd["rnn.weight_hh_l0"].shape == (G * H, H)
        seqs = opt.experiences_from_rollout(make_rollout(20, 3))
        l, e, g = opt.train(seqs)
        assert np.isfinite(float(l["loss"])) and np.isfinite(float(g["unclipped"]))


def test_masked_softmax_semantics():
    """policy.py:169-178: normalised over the mask, masked-out entries keep finite junk, empty rows -> +inf."""
    logits = torch.tensor([[[1.0, 2.0, 3.0], [0.5, 0.5, 0.5]]])
    mask = torch.tensor([[[True, False, True], [False, False, False]]])
    lp = masked_softmax(logits, mask)
    ref = torch.log_softmax(torch.tensor([1.0, 3.0]), 0)
    assert torch.allclose(lp[0, 0, [0, 2]], ref)
    assert torch.isfinite(lp[0, 0, 1])
    assert torch.isinf(lp[0, 1]).all()


def test_sample_index_function():
    logits = torch.tensor([0.1, 2.0, -1.0, 0.3])
    mask = torch.tensor([True, False, True, True])
    p = torch.softmax(logits[mask], 0).numpy()
    edges = np.cumsum(p)
    valid = [0, 2, 3]
    for u in (0.0, 0.1, 0.3, 0.5, 0.9, 0.999):
        assert sample_index(logits, mask, u) == valid[int(np.searchsorted(edges, u, side="right").clip(0, 2))]


# ------------------------------------------------------------------------------------------------ N-rank oracle
def test_nrank_oracle_matches_reference_under_gloo():
    """oracle/ref_distributed.py (one-process emulation) == 2 gloo processes running the reference's wrapper (recorded in
    tests/golden/reference_gloo_world2.npz).  The emulation performs the float32 sums of gloo's two-rank all-reduce, so
    the final weights of both ranks match the recording bit for bit."""
    from oracle import ref_distributed
    golden = _load_golden("reference_gloo_world2.npz")
    torch.set_num_threads(1)
    opts = [_oracle(8) for _ in range(2)]
    shards = [opts[r].experiences_from_rollout(make_rollout(24, 300 + r)) for r in range(2)]
    mine = [ref_distributed.train_ranks(opts, shards) for _ in range(2)]
    for r in range(2):
        for ep in range(2):
            l, e, g = mine[ep][r]
            got = [float(l[k]) for k in ("loss", "policy_loss", "entropy_loss", "value_loss")]
            np.testing.assert_array_equal(np.array(got), golden["rank%d_losses" % r][ep])
            np.testing.assert_allclose(float(g["unclipped"]), golden["rank%d_grad_norms" % r][ep][0], rtol=1e-6)
            np.testing.assert_allclose(float(g["clipped"]), golden["rank%d_grad_norms" % r][ep][1], rtol=1e-6)
        _assert_state_dict_matches(opts[r].policy_base.state_dict(), golden, "rank%d_final_" % r)


def test_target_unit_head_is_linear_in_the_unit_embedding():
    """Algebra behind DESIGN.md section 9 item 1 (checked on the CPU so the round-2 kernels have a pinned target):
    logits[n,u] = <att[n], W_g basic[n,u] + b_g> = <att[n] W_g, basic[n,u]> + <att[n], b_g>   (policy.py:101-131,152-153)
    and d_att[n] = W_g (sum_u dl[n,u] basic[n,u]) + (sum_u dl[n,u]) b_g -- neither needs the [N,40,128] embedding."""
    g = torch.Generator().manual_seed(5)
    N, units = 37, (1, 5, 16, 16, 1, 1)
    att = torch.randn(N, 128, generator=g, dtype=torch.float64).requires_grad_(True)
    basics = [torch.relu(torch.randn(N, n, 128, generator=g, dtype=torch.float64)) for n in units]
    Ws = [torch.randn(128, 128, generator=g, dtype=torch.float64) * 0.1 for _ in units]
    bs = [torch.randn(128, generator=g, dtype=torch.float64) * 0.1 for _ in units]
    ue = torch.cat([b @ W.t() + bias for b, W, bias in zip(basics, Ws, bs)], dim=1)          # [N, 40, 128]
    ref = torch.matmul(att.unsqueeze(-2), ue.transpose(-1, -2)).squeeze(-2)                    # policy.py:152-153
    dl = torch.randn(ref.shape, generator=g, dtype=torch.float64)
    (ref * dl).sum().backward()
    with torch.no_grad():
        logits, d_att, off = [], torch.zeros_like(att), 0
        for b, W, bias, n in zip(basics, Ws, bs, units):
            q = att @ W                                   # [N,128]: ONE small GEMM over tokens instead of n_u x as many rows
            c = att @ bias                                # [N]
            logits.append(torch.einsum("nc,nuc->nu", q, b) + c[:, None])
            P = torch.einsum("nu,nuc->nc", dl[:, off:off + n], b)
            d_att += P @ W.t() + dl[:, off:off + n].sum(1, keepdim=True) * bias
            off += n
        torch.testing.assert_close(torch.cat(logits, dim=1), ref.detach(), rtol=1e-10, atol=1e-10)
        torch.testing.assert_close(d_att, att.grad, rtol=1e-10, atol=1e-10)


def test_unit_encoder_backward_without_the_embedding_gradient():
    """Algebra and index arithmetic behind the fused unit-encoder backward (csrc/gemm_tf32x3.cu: dc_unit_wgrad_routed,
    dc_unit_dgrad_fused), restated in numpy with the kernels' own tiling -- 125-row tiles / 30-row K-chunks of whole tokens for
    the 5-unit group -- against torch autograd through the materialised [N,40,128] embedding (policy.py:99-136,144-153):
      dW_g = R^T basic_g + att^T s_g,  db_g = colsum R + att^T sum_u dlogits,   R = max-pool routing, s_g = sum_u dlogits_u basic_u
      dW_b = sum_g (relu' . ((R + dlogits x att) W_g))^T units_g."""
    import torch.nn.functional as F
    UNITS, OFF, N, BM = (1, 5, 16, 16, 1, 1), (0, 1, 6, 22, 38, 39), 29, 128
    g = torch.Generator().manual_seed(1)
    dd = dict(generator=g, dtype=torch.float64)
    w_b = (torch.randn(128, 12, **dd) * 0.3).requires_grad_(True)
    b_b = (torch.randn(128, **dd) * 0.1).requires_grad_(True)
    units = [torch.randn(N, n, 12, **dd) for n in UNITS]
    W = [(torch.randn(128, 128, **dd) * 0.1).requires_grad_(True) for _ in UNITS]
    b = [(torch.randn(128, **dd) * 0.1).requires_grad_(True) for _ in UNITS]
    att = torch.randn(N, 128, **dd)
    basic = [F.relu(F.linear(u, w_b, b_b)) for u in units]
    emb = [F.linear(x, w, bb) for x, w, bb in zip(basic, W, b)]
    mx = [e.max(dim=-2) for e in emb]
    xm = [m[0] for m in mx]
    xm[5] = xm[3]                                                  # policy.py:127
    tu = torch.einsum("nc,nuc->nu", att, torch.cat(emb, dim=-2))
    g_x, g_tu = torch.randn(N, 768, **dd), torch.randn(N, 40, **dd)
    g_tu[::2] = 0
    ((torch.cat(xm, dim=-1) * g_x).sum() + (tu * g_tu).sum()).backward()

    dxm, dl, attn = g_x.numpy(), g_tu.numpy(), att.numpy()
    dw_b, db_b = np.zeros((128, 12)), np.zeros(128)
    for gi, (NU, off) in enumerate(zip(UNITS, OFF)):
        Wg, bas = W[gi].detach().numpy(), basic[gi].detach().numpy().reshape(N * NU, 128)
        un, am = units[gi].numpy().reshape(N * NU, 12), mx[gi][1].numpy()
        routed = gi < 5
        dx = dxm[:, gi * 128:(gi + 1) * 128] + (dxm[:, 640:768] if gi == 3 else 0) if routed else None
        # --- dc_unit_dgrad_fused: tiles of whole tokens, d_emb generated row by row, mask recomputed from the raw features
        tile_rows = BM - BM % NU
        tile_toks = tile_rows // NU
        for mb in range((N * NU + tile_rows - 1) // tile_rows):
            tok0, m0 = mb * tile_toks, mb * tile_rows
            demb = np.zeros((128, 128))
            for r in range(tile_rows):
                n, u = tok0 + r // NU, r % NU
                if n < N:
                    if routed:
                        demb[r] = np.where(am[n] == u, dx[n], 0.0) if NU > 1 else dx[n]
                    demb[r] += dl[n, off + u] * attn[n]
            acc = demb @ Wg
            for row in range(min(tile_rows, N * NU - m0)):
                pre = un[m0 + row] @ w_b.detach().numpy().T + b_b.detach().numpy()
                gval = np.where(pre > 0, acc[row], 0.0)
                dw_b += np.outer(gval, un[m0 + row])
                db_b += gval
        # --- dc_unit_wgrad_routed: K-chunks of whole tokens (30 rows + 2 zero rows for the 5-unit group)
        dW, db = np.zeros((128, 128)), np.zeros(128)
        if routed and NU > 1:
            tpc = 32 // NU
            rpc, T = tpc * NU, N * NU
            for ch in range((T + rpc - 1) // rpc):
                A, X = np.zeros((32, 128)), np.zeros((32, 128))
                for i in range(rpc):
                    n = ch * tpc + i // NU
                    if n < N:
                        A[i] = np.where(am[n] == i % NU, dx[n], 0.0)
                    if ch * rpc + i < min(T, ch * rpc + rpc):
                        X[i] = bas[ch * rpc + i]
                dW += A.T @ X
                db += A.sum(0)
        elif routed:
            dW, db = dx.T @ bas, dx.sum(0)
        s = np.einsum("nu,nuj->nj", dl[:, off:off + NU], bas.reshape(N, NU, 128))       # dc_target_unit_q_bwd
        dW, db = dW + attn.T @ s, db + attn.T @ dl[:, off:off + NU].sum(1)                # the head's share: one token-level product
        np.testing.assert_allclose(dW, W[gi].grad.numpy(), rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(db, b[gi].grad.numpy(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(dw_b, w_b.grad.numpy(), rtol=1e-9, atol=1e-9)
    np.testing.assert_allclose(db_b, b_b.grad.numpy(), rtol=1e-9, atol=1e-9)
