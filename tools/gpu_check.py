#!/usr/bin/env python
"""Developer diagnostic for a GPU box: ours vs CPU oracle vs the unmodified reference extension, the sort
against CUB, and rough timings.  Prints a full report instead of stopping at the first failure (the pytest
suite under tests/ is the formal gate; this is the flashlight)."""
import argparse
import os
import sys
import time
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests import common  # noqa: E402
from seganygaussians_b200 import synthetic, _lib  # noqa: E402


def section(t):
    print("\n" + "=" * 100 + "\n" + t + "\n" + "=" * 100, flush=True)


def parity(name, P, H, W, K, depth=False, use_sh=False, deg=0, M=0, with_oracle=True, with_ref=True):
    section(f"parity {name}: P={P} {H}x{W} K={K} depth={depth} sh={use_sh}")
    sc = synthetic.scene(P, H, W, K, sh_coeffs=M)
    res = {}
    try:
        ours = common.run_torch_impl("ours", sc, K, depth=depth, use_sh=use_sh, sh_degree=deg)
        vis = int((ours.radii > 0).sum())
        print(f"ours: vis={vis} R={ours.num_rendered} n_contrib mean={ours.n_contrib.mean():.1f}")
        if K == 32 and not depth:
            simt = common.run_torch_impl("ours", sc, K, depth=depth, use_sh=use_sh, sh_degree=deg, tensor_cores=False)
            simt.kind = "ours-simt"
            print("-- tensor-core path vs fp32 SIMT path:")
            common.compare(ours, simt)
    except Exception:
        traceback.print_exc()
        return False
    ok_all = True
    if with_oracle:
        try:
            orc = common.run_oracle(sc, K, depth=depth, use_sh=use_sh, sh_degree=deg, nthreads=8)
            ok, _ = common.compare(ours, orc)
            ok_all &= ok
        except Exception:
            traceback.print_exc()
            ok_all = False
    if with_ref and common.have_ref(common.variant_of(K, depth)):
        try:
            ref = common.run_torch_impl("ref", sc, K, depth=depth, use_sh=use_sh, sh_degree=deg)
            ok, _ = common.compare(ours, ref, ints=common.INT_FWD, floats=common.FLOAT_FWD + common.GRADS +
                                   ("means2D", "conic_opacity", "depths", "cov3D"))
            ok_all &= ok
            if with_oracle:
                print("-- oracle vs reference (pins the oracle):")
                ok2, _ = common.compare(orc, ref)
            ref2 = common.run_torch_impl("ref", sc, K, depth=depth, use_sh=use_sh, sh_degree=deg)
            print("-- reference vs reference (run-to-run atomics noise):")
            common.compare(ref2, ref, ints=(), floats=common.GRADS)
        except Exception:
            traceback.print_exc()
            ok_all = False
    return ok_all


def sort_check():
    section("sort: own radix vs CUB vs torch.sort(stable)")
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    ok_all = True
    for n, bits in [(1, 41), (255, 41), (4096, 45), (4097, 46), (100003, 45), (3000000, 45), (1000000, 33), (50000, 64)]:
        g = torch.Generator().manual_seed(n)
        hi = torch.randint(0, 1 << min(bits - 32, 13), (n,), generator=g, dtype=torch.int64) if bits > 32 else torch.zeros(n, dtype=torch.int64)
        lo = torch.randint(0, 1 << 20, (n,), generator=g, dtype=torch.int64)  # many ties -> stability matters
        keys = ((hi << 32) | lo).to(dev)
        vals = torch.arange(n, dtype=torch.int32, device=dev)
        temp = torch.empty(int(lib.sagars_sort_temp_bytes(n)), dtype=torch.uint8, device=dev)
        outs = []
        for use_cub in (0, 1):
            ko = torch.empty_like(keys)
            vo = torch.empty_like(vals)
            rc = lib.sagars_sort_pairs(0, n, bits, keys.data_ptr(), vals.data_ptr(), ko.data_ptr(), vo.data_ptr(),
                                       temp.data_ptr(), use_cub, torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            if rc != 0:
                print("  sort rc", rc, _lib.last_error())
            outs.append((ko.clone(), vo.clone()))
        mask = (1 << bits) - 1 if bits < 63 else -1
        sk, idx = torch.sort(keys & mask if bits < 63 else keys, stable=True)
        ref_v = vals[idx]
        e_own = bool(torch.equal(outs[0][0], keys[idx]) and torch.equal(outs[0][1], ref_v))
        e_cub = bool(torch.equal(outs[1][0], keys[idx]) and torch.equal(outs[1][1], ref_v))
        ok_all &= e_own
        print(f"  n={n:8d} bits={bits}: own==torch {e_own}  cub==torch {e_cub}")
    return ok_all


def timing(P, H, W, K, iters=10, depth=False, use_sh=False, deg=0, M=0):
    section(f"timing: P={P} {H}x{W} K={K} depth={depth} sh={use_sh}")
    dev = torch.device("cuda", 0)
    sc = synthetic.scene(P, H, W, K, sh_coeffs=M)
    variant = common.variant_of(K, depth)
    from seganygaussians_b200 import rasterizer as R
    impls = {"ours": (R.GaussianRasterizationSettings, {"base": R.GaussianRasterizer, "cf": R.GaussianRasterizerContrastiveF,
                                                        "depth": R.GaussianRasterizerDepth}[variant])}
    if common.have_ref(variant):
        m = common.ref_module(variant)
        impls["ref"] = (m.GaussianRasterizationSettings, m.GaussianRasterizer)
    g = sc.gauss
    dL = sc.dL_dout[:K].to(dev)
    for name, (Settings, Rast) in impls.items():
        L = common._leafs(sc, dev, use_sh)
        rs = common._settings(Settings, sc, dev, K, deg)
        rast = Rast(raster_settings=rs)

        def step():
            for t in (L.means3D, L.means2D, L.opacities, L.scales, L.rotations, L.colors, L.shs, getattr(L, "mask", None)):
                if t is not None:
                    t.grad = None
            kw = dict(means3D=L.means3D, means2D=L.means2D, opacities=L.opacities, shs=L.shs,
                      colors_precomp=L.colors, scales=L.scales, rotations=L.rotations, cov3D_precomp=None)
            if depth:
                color, om, od, radii = rast(mask=L.mask, **kw)
            else:
                color, radii = rast(**kw)
            return color

        for _ in range(3):
            c = step(); c.backward(dL)
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tf = tb = 0.0
        for _ in range(iters):
            e[0].record(); c = step(); e[1].record(); c.backward(dL); e[2].record()
            torch.cuda.synchronize()
            tf += e[0].elapsed_time(e[1]); tb += e[1].elapsed_time(e[2])
        R_ = int(c.grad_fn.num_rendered) if hasattr(c.grad_fn, "num_rendered") else -1
        print(f"  {name:5s}: fwd {tf / iters:8.3f} ms  bwd {tb / iters:8.3f} ms  total {(tf + tb) / iters:8.3f} ms   R={R_}"
              f"  -> {P * H * W / ((tf + tb) / iters * 1e-3) / 1e12:.3f} T Gaussian*pixel/s", flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--tiny", action="store_true", help="only the smallest parity case (for compute-sanitizer)")
    ap.add_argument("--no-timing", action="store_true")
    ap.add_argument("--large", action="store_true", help="BASELINE-scale parity + timing of the other configs (c1, c3-like, c5-like)")
    a = ap.parse_args()
    print("device:", torch.cuda.get_device_name(0), "| lib:", _lib.load().sagars_arch().decode())
    results = {}
    if a.tiny:
        results["tiny_cf"] = parity("tiny_cf", 500, 40, 56, 32, with_ref=False)
        results["tiny_depth"] = parity("tiny_depth", 500, 40, 56, 3, depth=True, with_ref=False)
        print(results)
        sys.exit(0 if all(results.values()) else 1)
    if a.large:
        results["c1"] = parity("c1", 10000, 256, 256, 3, with_oracle=True)
        results["c3_like"] = parity("c3_like", 5000000, 1036, 1600, 32, with_oracle=False)
        results["c5_like"] = parity("c5_like", 2000000, 1600, 1600, 3, depth=True, use_sh=True, deg=3, M=16, with_oracle=False)
        timing(10000, 256, 256, 3)
        timing(5000000, 1036, 1600, 32, iters=5)
        timing(2000000, 1600, 1600, 3, iters=5, depth=True, use_sh=True, deg=3, M=16)
        timing(1000000, 1080, 1920, 3, iters=5)
        section("summary")
        for k, v in results.items():
            print(f"  {k:14s} {'OK' if v else 'FAIL'}")
        sys.exit(0 if all(results.values()) else 1)
    results["sort"] = sort_check()
    results["cf_small"] = parity("cf_small", 3000, 72, 104, 32)
    results["base_small"] = parity("base_small", 3000, 72, 104, 3)
    results["depth_small"] = parity("depth_small", 3000, 72, 104, 3, depth=True)
    results["base_sh"] = parity("base_sh", 2000, 64, 80, 3, use_sh=True, deg=3, M=16)
    results["depth_sh"] = parity("depth_sh", 2000, 64, 80, 3, depth=True, use_sh=True, deg=3, M=16)
    results["cf_medium"] = parity("cf_medium", 200000, 540, 960, 32)
    results["cf_c2"] = parity("cf_c2", 1000000, 1080, 1920, 32, with_oracle=False)
    if not a.no_timing:
        timing(1000000, 1080, 1920, 32)
        timing(10000, 256, 256, 3)
    section("summary")
    for k, v in results.items():
        print(f"  {k:14s} {'OK' if v else 'FAIL'}")
