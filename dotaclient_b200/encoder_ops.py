"""Autograd wrappers of the unit encoder and the target-unit head (``policy.py:99-136,144-153``).

Forward and backward are explicit chains of C-ABI kernels -- the fp32-accurate tensor-core GEMMs of
``csrc/gemm_tf32x3.cu`` for the 128x128 unit embeddings and the bandwidth kernels of ``csrc/encoder.cu`` around them --
neither pass materialises the [N, 40, 128] unit embedding or its gradient: forward has the max-pool in the embedding GEMM's
epilogue and the target-unit head through ``att W_g``; backward generates the max-pool routing inside the weight- and
data-gradient kernels and takes the head's rank-1 share through token-level products.
"""
import torch

from . import _lib
from .ops import PROFILE, _f32c, _need_cuda, gemm_tf32x3, gemm_wgrad_supported, wait_h2d

UNITS = (1, 5, 16, 16, 1, 1)              # allied/enemy heroes, allied/enemy non-heroes, allied/enemy towers
OFFSETS = (0, 1, 6, 22, 38, 39)
MAX_UNITS = 40
C = 128
XCAT = 7 * C                               # pre-rnn input row: env encoding + six group maxima (policy.py:129-136)

_basic_ws = {}


def _basic_workspace(device):
    ws = _basic_ws.get(device)
    if ws is None:
        ws = torch.empty(int(_lib.load().dc_unit_basic_bwd_workspace_bytes()), dtype=torch.uint8, device=device)
        _basic_ws[device] = ws
    return ws


_env_ws = {}


def _env_workspace(device):
    ws = _env_ws.get(device)
    if ws is None:
        ws = torch.empty(int(_lib.load().dc_env_bwd_workspace_bytes()), dtype=torch.uint8, device=device)
        _env_ws[device] = ws
    return ws


_wgrad_ws = {}


def _wgrad_workspace(No, Ni, device):
    key = (No, Ni, device)
    ws = _wgrad_ws.get(key)
    if ws is None:
        ws = torch.empty(int(_lib.load().dc_gemm_wgrad_workspace_bytes(No, Ni)), dtype=torch.uint8, device=device)
        _wgrad_ws[key] = ws
    return ws


# The unit embedding [N, 40, 128] (policy.py:130-131) is never materialised in the forward pass.  Its two consumers are
#   * the max-pool: fused into the epilogue of the embedding GEMM (dc_gemm_unit_max: max + arg-max per token and channel; the
#     1-unit groups are plain GEMMs writing their slot of the pre-rnn row; the enemy-tower embedding is not needed at all in
#     forward because policy.py:127 takes that slot's maximum from the enemy non-heroes);
#   * the target-unit head, which is linear in it: logits[n,u] = <att[n] W_g, basic[n,u]> + <att[n], b_g>  (TargetUnit below).
# In backward the embedding's gradient d_emb[n,u,:] has two sources -- the head (rank 1: dlogits[n,u] * att[n,:], arrives first) and the
# max-pool routing R (d_xmax[n,:] to the arg-max unit of every channel; arrives with the pre-rnn gradient, after the recurrence).
# TargetUnit parks (dlogits, att, s) in the `link` cell the two Functions of one graph share; UnitEncoder.backward then needs no
# dense [N, 40, 128] tensor at all:
#   dW_g  = R^T basic_g  (dc_unit_wgrad_routed: R generated in the A producer)  +  att^T s_g   (one token-level GEMM for all groups,
#           s_g = sum_u dlogits_u basic_u from dc_target_unit_q_bwd; its bias block gives the head's share of db_g)
#   dW_b += (relu'(.) (R + dlogits x att) W_g)^T units   (dc_unit_dgrad_fused_mask: d_emb generated in the producers, the ReLU mask
#           read as the bits the forward stored next to `basic`, dW_b reduced in the epilogue) -- d_basic never exists either.


def _ptr(t, float_offset=0):
    return t.data_ptr() + 4 * float_offset


def _ptr6(tensors):
    return (_lib._c.c_void_p * 6)(*[t.data_ptr() for t in tensors])


class UnitEncoder(torch.autograd.Function):
    """(env, w_e, b_e, w_b, b_b, units x6, W_g x6, b_g x6) -> the pre-rnn input row ``[..., 896]`` = relu(affine_env(env))
    followed by the six group maxima, written in place by the kernels (no cat, no ``[N, 40, 128]`` embedding).

    maxima slot 5 (enemy towers) is a copy of slot 3 (enemy non-heroes): the reference's ``policy.py:127``.
    ``link`` (a dict) receives the per-group ``basic`` activations and the embedding weights for the target-unit head.
    """

    @staticmethod
    def forward(ctx, link, keep_mask, env, w_e, b_e, w_b, b_b, *rest):
        units, weights, biases = rest[:6], rest[6:12], rest[12:18]
        ctx.link = link
        _need_cuda(env, w_b, *units)
        lib = _lib.load()
        st = _lib.stream_ptr()
        lead = units[0].shape[:-2]
        N = 1
        for d in lead:
            N *= d
        dev = units[0].device
        w_b, b_b = _f32c(w_b.detach()), _f32c(b_b.detach())
        units = [_f32c(u.detach()).reshape(N * n, 12) for u, n in zip(units, UNITS)]
        units = [u if u.data_ptr() % 16 == 0 else u.clone() for u in units]   # the backward kernels read whole rows as 3 x 16 bytes
        weights = [_f32c(w.detach()) for w in weights]
        biases = [_f32c(b.detach()) for b in biases]
        xcat = torch.empty((N, XCAT), dtype=torch.float32, device=dev)
        argmax = torch.zeros((5, N, C), dtype=torch.uint8, device=dev)         # 1-unit groups: the maximum is unit 0
        env2 = _f32c(env.detach()).reshape(N, 3)
        w_e, b_e = _f32c(w_e.detach()), _f32c(b_e.detach())
        wait_h2d(env2)
        with PROFILE.span("env_fwd", 1, 4 * N * (3 + C)):
            _lib.check(lib.dc_env_fwd(env2.data_ptr(), w_e.data_ptr(), b_e.data_ptr(), xcat.data_ptr(), XCAT, N, st), "dc_env_fwd")
        basics, masks = [], []
        for g, n_u in enumerate(UNITS):
            R = N * n_u
            basic = torch.empty((R, C), dtype=torch.float32, device=dev)
            wait_h2d(units[g])                       # this group's observations may still be in flight over PCIe
            if keep_mask:                            # the ReLU sign bits of `basic` for the backward: 1/32 of its bytes
                mask = torch.empty(((R + 31) // 32, C), dtype=torch.int32, device=dev)
                with PROFILE.span("unit_basic_fwd", 1, 4 * R * (12 + C) + mask.numel() * 4):
                    _lib.check(lib.dc_unit_basic_fwd_mask(units[g].data_ptr(), w_b.data_ptr(), b_b.data_ptr(), basic.data_ptr(),
                                                          mask.data_ptr(), R, st), "dc_unit_basic_fwd_mask")
                masks.append(mask)
            else:
                with PROFILE.span("unit_basic_fwd", 1, 4 * R * (12 + C)):
                    _lib.check(lib.dc_unit_basic_fwd(units[g].data_ptr(), w_b.data_ptr(), b_b.data_ptr(), basic.data_ptr(), R, st),
                               "dc_unit_basic_fwd")
            if n_u > 1:                               # embedding GEMM with the max-pool in its epilogue
                copy = _ptr(xcat, 6 * C) if g == 3 else None
                with PROFILE.span("gemm_unit_max", 1, 4 * (R * C + C * C + N * C) + N * C):
                    _lib.check(lib.dc_gemm_unit_max(basic.data_ptr(), weights[g].data_ptr(), biases[g].data_ptr(),
                                                    _ptr(xcat, (g + 1) * C), copy, XCAT, argmax[g].data_ptr(), N, n_u, st),
                               "dc_gemm_unit_max")
            elif g < 5:                               # one unit: the embedding IS the maximum -> straight into its slot
                with PROFILE.span("gemm_tf32x3", 1, 4 * (2 * R * C + C * C)):
                    _lib.check(lib.dc_gemm_tf32x3_blocked(basic.data_ptr(), C, 0, 0, weights[g].data_ptr(), C, biases[g].data_ptr(),
                                                          _ptr(xcat, (g + 1) * C), XCAT, 0, 0, R, C, C, 0, st), "dc_gemm_tf32x3_blocked")
            basics.append(basic)
        link["basics"], link["weights"], link["biases"] = basics, weights, biases
        ctx.N = N
        ctx.lead = lead
        ctx.keep_mask = keep_mask
        ctx.save_for_backward(argmax, *units, *basics, *weights, env2, xcat, *masks)
        return xcat.view(*lead, XCAT)

    @staticmethod
    def backward(ctx, d_xcat):
        saved = ctx.saved_tensors
        argmax, units, basics, weights, env2, xcat = saved[0], saved[1:7], saved[7:13], saved[13:19], saved[19], saved[20]
        masks = saved[21:27]
        N = ctx.N
        lib = _lib.load()
        st = _lib.stream_ptr()
        dev = argmax.device
        pending = ctx.link.pop("pending", None)
        d_xcat = _f32c(d_xcat).reshape(N, XCAT)
        dw_e = torch.empty((C, 3), dtype=torch.float32, device=dev)
        db_e = torch.empty(C, dtype=torch.float32, device=dev)
        with PROFILE.span("env_bwd", 2, 4 * N * (2 * C + 3)):
            _lib.check(lib.dc_env_bwd(d_xcat.data_ptr(), xcat.data_ptr(), XCAT, env2.data_ptr(), dw_e.data_ptr(), db_e.data_ptr(),
                                      N, _env_workspace(dev).data_ptr(), st), "dc_env_bwd")
        dl = att = s_head = None
        if pending is not None:
            dl, att, s_head = pending
        dw_b = db_b = None                              # the forward kept the ReLU mask iff w_b / b_b need a gradient
        if ctx.keep_mask:
            dw_b = torch.empty((C, 12), dtype=torch.float32, device=dev)
            db_b = torch.empty(C, dtype=torch.float32, device=dev)
        dw_all = torch.zeros((6, C, C), dtype=torch.float32, device=dev)     # zeros: the enemy-tower layer has no max-pool path
        db_all = torch.zeros((6, C), dtype=torch.float32, device=dev)
        ws_w = _wgrad_workspace(C, C, dev)
        ws_b = _basic_workspace(dev)
        for g, (n_u, off) in enumerate(zip(UNITS, OFFSETS)):
            R = N * n_u
            routed = g < 5                                 # policy.py:127: enemy towers never reach the maxima
            dx = _ptr(d_xcat, (g + 1) * C) if routed else None
            dx2 = _ptr(d_xcat, 6 * C) if g == 3 else None  # ... their slot was fed from the enemy non-hero maximum
            if routed and n_u > 1:
                with PROFILE.span("gemm_wgrad", 2, 4 * (R * C + C * C + N * C) + N * C):   # dW_g = R^T basic_g, db_g = colsum(R)
                    _lib.check(lib.dc_unit_wgrad_routed(dx, dx2, XCAT, argmax[g].data_ptr(), basics[g].data_ptr(), N, n_u,
                                                        dw_all[g].data_ptr(), db_all[g].data_ptr(), ws_w.data_ptr(), st),
                               "dc_unit_wgrad_routed")
            elif routed:                                   # one unit: the routing is the gradient of the maximum itself
                with PROFILE.span("gemm_wgrad", 2, 4 * (2 * R * C + C * C)):
                    _lib.check(lib.dc_gemm_wgrad_tf32x3(dx, XCAT, basics[g].data_ptr(), C, R, C, C, dw_all[g].data_ptr(), C,
                                                        db_all[g].data_ptr(), 0, ws_w.data_ptr(), st), "dc_gemm_wgrad_tf32x3")
            if not ctx.keep_mask:
                continue
            wt = weights[g].t().contiguous()
            with PROFILE.span("unit_dgrad_fused", 2, N * (4 * C + C) * (1 if routed else 0) + 4 * R * 12 + masks[g].numel() * 4 +
                              (4 * N * (C + n_u) if dl is not None else 0)):
                _lib.check(lib.dc_unit_dgrad_fused_mask(dx, dx2, XCAT, argmax[g].data_ptr() if (routed and n_u > 1) else None,
                                                        None if dl is None else _ptr(dl, off), MAX_UNITS,
                                                        None if att is None else att.data_ptr(), wt.data_ptr(), units[g].data_ptr(),
                                                        masks[g].data_ptr(), N, n_u, dw_b.data_ptr(), db_b.data_ptr(), 1 if g > 0 else 0,
                                                        ws_b.data_ptr(), st), "dc_unit_dgrad_fused_mask")
        if dl is not None:
            # the head's share of every dW_g and db_g in ONE token-level product: att^T [s_0 | ... | s_5 | sum_u dlogits]
            dw_head = torch.empty((C, QW), dtype=torch.float32, device=dev)
            with PROFILE.span("gemm_wgrad", 2, 4 * (N * C + N * QW + C * QW)):
                _lib.check(lib.dc_gemm_wgrad_tf32x3(att.data_ptr(), C, s_head.data_ptr(), QW, N, C, QW, dw_head.data_ptr(), QW, None, 0,
                                                    _wgrad_workspace(C, QW, dev).data_ptr(), st), "dc_gemm_wgrad_tf32x3")
            dw_all += dw_head[:, :6 * C].reshape(C, 6, C).permute(1, 0, 2)
            db_all += dw_head[:, 6 * C:6 * C + 6].t()
        dws, dbs = list(dw_all.unbind(0)), list(db_all.unbind(0))
        return (None, None, None, dw_e, db_e, dw_b, db_b) + (None,) * 6 + tuple(dws) + tuple(dbs)


QW = 7 * C     # width of the head's token-level operands: six groups x 128 channels + one block carrying the six bias dots


class TargetUnit(torch.autograd.Function):
    """``logits[..., u] = <attention, unit_embedding[..., u, :]>`` (``policy.py:152-153``) WITHOUT the embedding:
    ``<att, W_g basic_u + b_g> = <att W_g, basic_u> + <att, b_g>``.  One GEMM over tokens produces ``q = att [W_0|..|W_5|b]``
    ``[N, 896]``, a bandwidth kernel dots it with the stored ``basic`` rows.  Backward: ``s_g = sum_u dlogits_u basic_u`` (same
    kernel shape), ``d_att = s [W_0|..|W_5|b]^T`` (one GEMM); the gradient towards the embedding weights and the basic layer
    is finished by ``UnitEncoder.backward`` from (dlogits, att, s) parked in ``link``."""

    @staticmethod
    def forward(ctx, att, link):
        _need_cuda(att)
        basics, weights, biases = link["basics"], link["weights"], link["biases"]
        lead = att.shape[:-1]
        N = att.numel() // C
        att2 = _f32c(att.detach()).reshape(N, C)
        dev = att2.device
        bias_block = torch.zeros((C, C), dtype=torch.float32, device=dev)
        bias_block[:, :6] = torch.stack(biases, dim=1)
        bm = torch.cat(list(weights) + [bias_block], dim=1)                  # [128, 896]: bm[c, g*128+j] = W_g[c,j], bm[c, 768+g] = b_g[c]
        q = gemm_tf32x3(att2, bm.t().contiguous())                           # [N, 896] = att [W_0 | ... | W_5 | b]
        logits = torch.empty((N, MAX_UNITS), dtype=torch.float32, device=dev)
        with PROFILE.span("target_unit_fwd", 1, 4 * N * (MAX_UNITS * C + QW + MAX_UNITS)):
            _lib.check(_lib.load().dc_target_unit_q_fwd(q.data_ptr(), QW, _ptr6(basics), logits.data_ptr(), N, _lib.stream_ptr()),
                       "dc_target_unit_q_fwd")
        ctx.save_for_backward(att2, bm, *basics)
        ctx.link = link
        ctx.att_shape = att.shape
        return logits.view(*lead, MAX_UNITS)

    @staticmethod
    def backward(ctx, dlogits):
        att2, bm = ctx.saved_tensors[:2]
        basics = ctx.saved_tensors[2:]
        N = att2.shape[0]
        dl = _f32c(dlogits).reshape(N, MAX_UNITS)
        s = torch.empty((N, QW), dtype=torch.float32, device=att2.device)
        with PROFILE.span("target_unit_bwd", 1):       # bytes depend on how many tokens used the head (others are skipped)
            _lib.check(_lib.load().dc_target_unit_q_bwd(dl.data_ptr(), _ptr6(basics), s.data_ptr(), QW, N, _lib.stream_ptr()),
                       "dc_target_unit_q_bwd")
        d_att = gemm_tf32x3(s, bm)                                          # [N, 128] = s [W_0 | ... | W_5 | b]^T
        ctx.link["pending"] = (dl, att2, s)                                  # consumed by UnitEncoder.backward
        return d_att.view(ctx.att_shape), None


def unit_encoder(env, w_e, b_e, w_b, b_b, units, weights, biases):
    """-> (``link``: the handle ``target_unit`` needs, pre-rnn input ``[..., 896]``)."""
    link = {}
    keep_mask = torch.is_grad_enabled() and (w_b.requires_grad or b_b.requires_grad)
    xcat = UnitEncoder.apply(link, keep_mask, env, w_e, b_e, w_b, b_b, *units, *weights, *biases)
    return link, xcat


def target_unit(att, link):
    return TargetUnit.apply(att, link)


__all__ = ["unit_encoder", "target_unit", "gemm_wgrad_supported"]
