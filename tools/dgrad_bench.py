"""Kernel-level timer of the unit-encoder data gradient (dc_unit_dgrad_fused and dc_unit_dgrad_fused_mask) on the C2 shapes.

The six calls of one UnitEncoder.backward at N = 131072 tokens (256 sequences x 512 steps): groups of 1, 5, 16, 16, 1 and 1
units, the max-pool routing on the first five groups (d_xmax read from the [N, 896] pre-rnn gradient), the second routing
source on group 3 (enemy non-heroes, which also feed the enemy-tower slot), the target-unit head terms on all six.

Each group is launched --iters times back to back between two CUDA events after --warmup launches.  One launch reads at least
150 MB (the d_xmax slice, att, dlogits, units), more than the 126 MB L2, so consecutive launches do not run from L2.
Per launch: microseconds and SM cycles per 128-row tile of the busiest CTA (ceil(tiles / SMs) tiles), at the SM clock
nvidia-smi reports while the launches run.

  python tools/dgrad_bench.py [--lib path/to/libdotaclient_b200.so ...] [--iters 300]

Several --lib give one table per library (e.g. two builds of the same tree), in the same process and on the same inputs.
"""
import argparse
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from dotaclient_b200 import _lib  # noqa: E402

UNITS = (1, 5, 16, 16, 1, 1)
OFFSETS = (0, 1, 6, 22, 38, 39)
C, XCAT, MAX_UNITS, KIN = 128, 896, 40, 12


def load(path):
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SIGNATURES.items():
        if hasattr(lib, name):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
    return lib


def check(lib, rc, what):
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (what, rc, lib.dc_last_error().decode()))


def smi(fields):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=" + fields,
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        return [s.strip() for s in out.strip().split(",")]
    except (OSError, subprocess.SubprocessError):
        return None


def make_inputs(N, dev, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    t = dict(
        units=[torch.randn(N * n, KIN, generator=g).to(dev) for n in UNITS],
        w_b=(torch.randn(C, KIN, generator=g) * 0.3).to(dev),
        b_b=(torch.randn(C, generator=g) * 0.1).to(dev),
        wt=[(torch.randn(C, C, generator=g) * 0.09).to(dev) for _ in UNITS],
        d_xcat=torch.randn(N, XCAT, generator=g).to(dev),
        argmax=torch.stack([torch.randint(0, n, (N, C), generator=g, dtype=torch.uint8) for n in UNITS[:5]]).to(dev),
        dl=torch.randn(N, MAX_UNITS, generator=g).to(dev),
        att=torch.randn(N, C, generator=g).to(dev),
    )
    return t


def launches(lib, t, N, with_mask, masks, ws, dwb, dbb, st):
    """-> one closure per group issuing that group's data-gradient call exactly as UnitEncoder.backward does."""
    dx_base = t["d_xcat"].data_ptr()
    calls = []
    for g, (n_u, off) in enumerate(zip(UNITS, OFFSETS)):
        routed = g < 5
        dx = dx_base + 4 * (g + 1) * C if routed else None
        dx2 = dx_base + 4 * 6 * C if g == 3 else None
        am = t["argmax"][g].data_ptr() if (routed and n_u > 1) else None
        head = (t["dl"].data_ptr() + 4 * off, MAX_UNITS, t["att"].data_ptr(), t["wt"][g].data_ptr(), t["units"][g].data_ptr())
        acc = 1 if g > 0 else 0
        if with_mask:
            args = (dx, dx2, XCAT, am) + head + (masks[g].data_ptr(), N, n_u, dwb.data_ptr(), dbb.data_ptr(), acc, ws.data_ptr(), st)
            calls.append(lambda a=args: check(lib, lib.dc_unit_dgrad_fused_mask(*a), "dc_unit_dgrad_fused_mask"))
        else:
            args = (dx, dx2, XCAT, am) + head + (t["w_b"].data_ptr(), t["b_b"].data_ptr(), N, n_u, dwb.data_ptr(), dbb.data_ptr(), acc,
                                                 ws.data_ptr(), st)
            calls.append(lambda a=args: check(lib, lib.dc_unit_dgrad_fused(*a), "dc_unit_dgrad_fused"))
    return calls


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--lib", action="append", default=None, help="library to time (default: the in-tree build); repeatable")
    p.add_argument("--tokens", type=int, default=131072)
    p.add_argument("--iters", type=int, default=300)
    p.add_argument("--warmup", type=int, default=20)
    a = p.parse_args()
    assert torch.cuda.is_available(), "dgrad_bench needs a GPU"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    libs = a.lib or [_lib.LIB_PATH]
    info = smi("name,power.limit,clocks.max.sm")
    print("card: %s, power limit %s W, max SM clock %s MHz" % tuple(info) if info else "card: nvidia-smi unavailable")
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    N = a.tokens
    t = make_inputs(N, dev)
    st = torch.cuda.current_stream().cuda_stream
    dwb, dbb = torch.empty(C, KIN, device=dev), torch.empty(C, device=dev)
    for path in libs:
        lib = load(path)
        ws = torch.empty(int(lib.dc_unit_basic_bwd_workspace_bytes()), dtype=torch.uint8, device=dev)
        masks = None
        if hasattr(lib, "dc_unit_basic_fwd_mask"):
            masks = []
            for g, n_u in enumerate(UNITS):
                R = N * n_u
                basic = torch.empty(R, C, device=dev)
                m = torch.empty((R + 31) // 32, C, dtype=torch.int32, device=dev)
                check(lib, lib.dc_unit_basic_fwd_mask(t["units"][g].data_ptr(), t["w_b"].data_ptr(), t["b_b"].data_ptr(),
                                                      basic.data_ptr(), m.data_ptr(), R, st), "dc_unit_basic_fwd_mask")
                masks.append(m)
            del basic
        entries = [("dc_unit_dgrad_fused", False)] + ([("dc_unit_dgrad_fused_mask", True)] if masks is not None else [])
        print("\n== %s" % os.path.relpath(os.path.abspath(path), ROOT))
        for name, with_mask in entries:
            calls = launches(lib, t, N, with_mask, masks, ws, dwb, dbb, st)
            for fn in calls:
                for _ in range(a.warmup):
                    fn()
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in calls]
            for fn, (e0, e1) in zip(calls, ev):
                e0.record()
                for _ in range(a.iters):
                    fn()
                e1.record()
            clk = smi("clocks.sm")                       # sampled while the queued launches run
            torch.cuda.synchronize()
            mhz = float(clk[0]) if clk else float("nan")
            total = 0.0
            print("%s  (SM clock %.0f MHz during the run)" % (name, mhz))
            print("  group units   rows      tiles  tiles/CTA   us/launch  cycles/tile")
            for g, (n_u, (e0, e1)) in enumerate(zip(UNITS, ev)):
                us = e0.elapsed_time(e1) * 1e3 / a.iters
                total += us
                rows = N * n_u
                tile_rows = 128 - 128 % n_u
                tiles = (rows + tile_rows - 1) // tile_rows
                per_cta = (tiles + n_sm - 1) // n_sm
                print("  %5d %5d %9d %8d %9d %11.1f %12.0f" % (g, n_u, rows, tiles, per_cta, us, us * mhz / per_cta))
            print("  all six groups: %.3f ms per backward" % (total / 1e3))


if __name__ == "__main__":
    main()
