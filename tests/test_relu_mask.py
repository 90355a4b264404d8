"""The ReLU sign mask the unit encoder's forward stores for its data gradient (dc_unit_basic_fwd_mask, dc_unit_dgrad_fused_mask).

Layout: uint32 [ceil(R/32), 128], bit i of word [b][j] = basic[32b + i][j] > 0, bits of rows >= R zero.  The data-gradient
kernel stages the words of one tile (128 rows, or 125 for the 5-unit group) and takes the 32 rows of each epilogue row group
from two neighbouring words and a funnel shift by the tile's first row mod 32.
"""
import importlib.util
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pack_mask(dense):
    """dense bool [R, 128] -> uint32 [ceil(R/32), 128] in the layout above."""
    R, C = dense.shape
    padded = np.zeros(((R + 31) // 32 * 32, C), dtype=np.uint64)
    padded[:R] = dense
    bits = padded.reshape(-1, 32, C) << np.arange(32, dtype=np.uint64)[None, :, None]
    return bits.sum(axis=1).astype(np.uint32)


def staged_row_bits(mask, R, tile_rows, tile, rng):
    """What the kernel's epilogue sees for one tile: for each 32-row group LD (0..3) the word of 32 mask bits of rows
    [32 LD, 32 LD + 32) of the tile.  Words are staged as in stage_units (first word m0 >> 5, as many as the tile's rows touch);
    the rest of the 5-word staging buffer holds stale data (random here)."""
    C = mask.shape[1]
    m0 = tile * tile_rows
    rows = min(tile_rows, R - m0)
    w0, w1 = m0 >> 5, (m0 + rows - 1) >> 5
    assert w1 - w0 + 1 <= 5
    staged = rng.integers(0, 2 ** 32, size=(5, C), dtype=np.uint64)
    staged[:w1 - w0 + 1] = mask[w0:w1 + 1]
    shift = m0 & 31
    out = []
    for LD in range(4):
        lo = staged[LD]
        if tile_rows < 128:
            hi = staged[LD + 1]
            out.append((((hi << np.uint64(32)) | lo) >> np.uint64(shift)) & np.uint64(0xFFFFFFFF))   # __funnelshift_r(lo, hi, shift)
        else:
            assert shift == 0
            out.append(lo)
    return out, rows


def test_mask_layout_matches_a_dense_sign_mask():
    rng = np.random.default_rng(0)
    for R in (1, 31, 32, 33, 1000, 5 * 1001):
        pre = rng.standard_normal((R, 128)).astype(np.float32)
        pre[rng.random((R, 128)) < 0.05] = 0.0                       # exact zeros are "off", like relu'(0) = 0
        dense = pre > 0
        mask = pack_mask(dense)
        assert mask.shape == ((R + 31) // 32, 128)
        for r in rng.integers(0, R, size=min(R, 200)):
            np.testing.assert_array_equal((mask[r // 32] >> np.uint32(r % 32)) & 1, dense[r])
        if R % 32:
            assert not np.any(mask[-1] >> np.uint32(R % 32))        # bits of rows past R are zero


@pytest.mark.parametrize("n_units", [1, 5, 16])
def test_tile_word_and_shift_arithmetic(n_units):
    """Every row of every tile, including the 125-row tiles whose 32-row groups straddle two words and a ragged last tile,
    reads its own bit through the staged words and the funnel shift."""
    rng = np.random.default_rng(n_units)
    tile_rows = 128 - 128 % n_units
    R = n_units * 1001                                              # 5-unit group: 40 whole tiles + a 5-row remainder
    dense = rng.random((R, 128)) < 0.5
    mask = pack_mask(dense)
    n_tiles = (R + tile_rows - 1) // tile_rows
    for tile in range(n_tiles):
        words, rows = staged_row_bits(mask, R, tile_rows, tile, rng)
        for LD in range(4):
            for jj in range(32):
                row = 32 * LD + jj
                if row < tile_rows and row < rows:
                    got = (words[LD] >> np.uint64(jj)) & np.uint64(1)
                    np.testing.assert_array_equal(got.astype(bool), dense[tile * tile_rows + row])


@pytest.fixture(scope="module")
def lib():
    from dotaclient_b200 import _lib, build
    build.build()
    return _lib.load()


def test_argument_errors_without_gpu(lib):
    """Both new entries validate their arguments before any CUDA call."""
    one = 4096                                       # any non-null, 16-byte aligned "pointer": validation fails before it is used
    assert lib.dc_unit_basic_fwd_mask(one, one, one, one, None, 8, None) == -1                        # no mask
    assert b"dc_unit_basic_fwd_mask" in lib.dc_last_error()
    assert lib.dc_unit_basic_fwd_mask(one, one, one, one, one + 4, 8, None) == -1                     # mask misaligned
    assert lib.dc_unit_basic_fwd_mask(one, one, one, one, one, 0, None) == -1                         # no rows
    args = [one, None, 896, one, None, 40, None, one, one, one, 8, 16, one, one, 0, one, None]
    bad = lambda i, v: lib.dc_unit_dgrad_fused_mask(*(args[:i] + [v] + args[i + 1:]))  # noqa: E731
    assert bad(9, None) == -1 and b"dc_unit_dgrad_fused_mask" in lib.dc_last_error()                # no mask
    assert bad(9, one + 4) == -1                                                                    # mask misaligned
    assert bad(7, None) == -1                                                                       # no W^T
    assert bad(11, 4) == -2                                                                         # 1, 5 or 16 units
    assert bad(3, None) == -1                                                                       # routing without arg-max
    assert bad(4, one) == -1                                                                        # dlogits without att
    assert bad(8, one + 4) == -1                                                                    # units misaligned
    assert b"dc_unit_dgrad_fused_mask" in lib.dc_last_error()


# ---------------------------------------------------------------------------------------------------------------------- GPU

def _encoder_check():
    spec = importlib.util.spec_from_file_location("encoder_check", os.path.join(ROOT, "tools", "encoder_check.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _forward_with_mask(lib, units, w_b, b_b):
    import torch
    from dotaclient_b200 import _lib
    R = units.shape[0]
    basic = torch.full((R, 128), 7.0, device=units.device)
    basic_m = torch.full((R, 128), 7.0, device=units.device)
    mask = torch.full(((R + 31) // 32, 128), -1, dtype=torch.int32, device=units.device)
    st = _lib.stream_ptr()
    _lib.check(lib.dc_unit_basic_fwd(units.data_ptr(), w_b.data_ptr(), b_b.data_ptr(), basic.data_ptr(), R, st), "dc_unit_basic_fwd")
    _lib.check(lib.dc_unit_basic_fwd_mask(units.data_ptr(), w_b.data_ptr(), b_b.data_ptr(), basic_m.data_ptr(), mask.data_ptr(), R, st),
               "dc_unit_basic_fwd_mask")
    return basic, basic_m, mask


@pytest.mark.gpu
@pytest.mark.parametrize("R", [1, 31, 32, 33, 5 * 1001, 131072 * 16])
def test_forward_mask_is_the_sign_of_basic(lib, R):
    """The mask equals basic > 0 bit for bit, and basic is the same with or without the mask output."""
    import torch
    dev = torch.device("cuda", 0)
    g = torch.Generator(device="cpu").manual_seed(R)
    units = torch.randn(R, 12, generator=g).to(dev)
    w_b, b_b = (torch.randn(128, 12, generator=g) * 0.3).to(dev), (torch.randn(128, generator=g) * 0.1).to(dev)
    basic, basic_m, mask = _forward_with_mask(lib, units, w_b, b_b)
    torch.cuda.synchronize()
    assert torch.equal(basic, basic_m)
    dense = (basic > 0).cpu().numpy()
    assert 0.2 < dense.mean() < 0.8
    np.testing.assert_array_equal(mask.cpu().numpy().view(np.uint32), pack_mask(dense))


def _dgrad_both(lib, t, N, n_u, dx2, head, routed, mask):
    """-> (dW_b, db_b) of dc_unit_dgrad_fused and of dc_unit_dgrad_fused_mask on the same inputs."""
    import torch
    from dotaclient_b200 import _lib
    dev, st = t["units"].device, _lib.stream_ptr()
    wt = t["W"].t().contiguous()
    ws = torch.empty(int(lib.dc_unit_basic_bwd_workspace_bytes()), dtype=torch.uint8, device=dev)
    dx = t["dx"].data_ptr()
    head_args = (dx + 4 * 256 if routed else None, dx + 4 * 640 if dx2 else None, 896,
                 t["am"].data_ptr() if (routed and n_u > 1) else None, t["dl"].data_ptr() + 4 * 3 if head else None, 40,
                 t["att"].data_ptr() if head else None, wt.data_ptr(), t["units"].data_ptr())
    out = []
    for use_mask in (False, True):
        dwb, dbb = torch.full((128, 12), 7.0, device=dev), torch.full((128,), 7.0, device=dev)
        if use_mask:
            _lib.check(lib.dc_unit_dgrad_fused_mask(*head_args, mask.data_ptr(), N, n_u, dwb.data_ptr(), dbb.data_ptr(), 0,
                                                    ws.data_ptr(), st), "dc_unit_dgrad_fused_mask")
        else:
            _lib.check(lib.dc_unit_dgrad_fused(*head_args, t["w_b"].data_ptr(), t["b_b"].data_ptr(), N, n_u, dwb.data_ptr(),
                                               dbb.data_ptr(), 0, ws.data_ptr(), st), "dc_unit_dgrad_fused")
        out.append((dwb, dbb))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("N,n_u,dx2,head,routed", [(1, 1, False, True, True), (7, 5, False, True, True), (130, 16, True, True, True),
                                                   (1000, 5, False, False, True), (1001, 16, False, True, True),
                                                   (300, 1, False, True, False), (26, 5, False, True, True)])
def test_dgrad_with_stored_mask_is_bit_identical(lib, N, n_u, dx2, head, routed):
    """dc_unit_dgrad_fused_mask == dc_unit_dgrad_fused bit for bit (same mask, every other line of the kernel shared), and both
    match the dense fp64 chain at the tolerances of the recomputing entry's own test."""
    import torch
    ec = _encoder_check()
    dev = torch.device("cuda", 0)
    inp, (_, _, dwb_r, dbb_r) = ec.dense_reference(N, n_u, 5 + N, dx2, head, routed)
    t = {k: v.to(dev).contiguous() for k, v in inp.items()}
    _, _, mask = _forward_with_mask(lib, t["units"], t["w_b"], t["b_b"])
    (dwb, dbb), (dwb_m, dbb_m) = _dgrad_both(lib, t, N, n_u, dx2, head, routed, mask)
    assert torch.equal(dwb, dwb_m) and torch.equal(dbb, dbb_m)
    tol = dict(rtol=1e-4, atol=2e-5 * max(1.0, float(dwb_r.abs().max())))
    torch.testing.assert_close(dwb_m.cpu().double(), dwb_r, **tol)
    torch.testing.assert_close(dbb_m.cpu().double(), dbb_r, **tol)


@pytest.mark.gpu
def test_dgrad_with_stored_mask_is_bit_identical_at_c2():
    """One 16-unit group at the benchmark's size (131072 tokens, both routing sources and the head): the two entries agree
    bit for bit."""
    import torch
    from dotaclient_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    N, n_u = 131072, 16
    g = torch.Generator(device="cpu").manual_seed(3)
    t = dict(units=torch.randn(N * n_u, 12, generator=g), w_b=torch.randn(128, 12, generator=g) * 0.3,
             b_b=torch.randn(128, generator=g) * 0.1, W=torch.randn(128, 128, generator=g) * 0.09, dx=torch.randn(N, 896, generator=g),
             am=torch.randint(0, n_u, (N, 128), generator=g, dtype=torch.uint8), dl=torch.randn(N, 40, generator=g),
             att=torch.randn(N, 128, generator=g))
    t = {k: v.to(dev).contiguous() for k, v in t.items()}
    _, _, mask = _forward_with_mask(lib, t["units"], t["w_b"], t["b_b"])
    (dwb, dbb), (dwb_m, dbb_m) = _dgrad_both(lib, t, N, n_u, True, True, True, mask)
    assert torch.equal(dwb, dwb_m) and torch.equal(dbb, dbb_m)
    assert float(dwb.abs().max()) > 0
