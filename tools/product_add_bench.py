"""Products with the error term (scgpu_*_add_batch) against their sibling call alone and against what a user composes
without them (sibling, then torch.remainder(out + e, q)), on the same seeded inputs, larger than L2 (2^20 rows, 2^19
instances of the Dilithium module shapes).  The three are timed in alternating rounds (CUDA events around `--calls`
calls each); the outputs of the fused call and of the composition are compared in full.  Rates are medians over the
rounds with their min / max; the HBM fraction counts the bytes the fused call must move (16 n per product, 12 n per
product against one shared key, 4 n (k l + l + 2 k) per module instance, 4 n (l + 2 k) against one shared matrix) over
7.7 TB/s.  The card's name and power limit are read in the same run.

usage: python tools/product_add_bench.py [--rounds 7] [--calls 3] [--out profiles/product_add_b200.json]"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

HBM = 7.7e12


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    except Exception as exc:                                  # the measurement stands without it; say so in the record
        return "unknown (%s)" % exc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--calls", type=int, default=3)
    ap.add_argument("--rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "product_add_b200.json"))
    args = ap.parse_args()

    import numpy as np
    import torch
    import _oracle as O
    import libsafecrypto_b200 as sc
    assert torch.cuda.is_available(), "this measurement needs a GPU"
    dev = "cuda:0"
    g = torch.Generator(device=dev).manual_seed(2026)

    def plan(q, n, in_range):
        w, r = O.tables(q, n, 16 if q < 32768 else 32)
        p = sc.NttPlan(n, q, sc.REFERENCE, w, r)
        if in_range:
            p.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        return p

    def rnd(lo, hi, shape):
        return torch.randint(lo, hi, shape, dtype=torch.int32, device=dev, generator=g)

    def shapes():
        rows = args.rows
        for q, n, in_range in ((12289, 512, False), (12289, 512, True), (12289, 1024, False), (8380417, 256, False)):
            p = plan(q, n, in_range)
            a, b, e = rnd(0, q, (rows, n)), rnd(0, q, (rows, n)), rnd(-8, 9, (rows, n))
            yield ("polymul q=%d n=%d%s" % (q, n, " in-range" if in_range else ""), q, rows, 16 * n, e,
                   lambda o, p=p, a=a, b=b: p.polymul(o, a, b), lambda o, p=p, a=a, b=b, e=e: p.polymul_add(o, a, b, e))
        p = plan(12289, 512, False)
        t, key, e = rnd(0, 12289, (rows, 512)), rnd(0, 12289, (512,)), rnd(-8, 9, (rows, 512))
        yield ("shared key q=12289 n=512", 12289, rows, 12 * 512, e,
               lambda o: p.mul_key(o, t, key), lambda o: p.mul_key_add(o, t, key, e))
        for q, k, l, cnt in ((7681, 3, 3, rows), (8380417, 5, 4, rows // 2)):
            pm = plan(q, 256, False)
            A, s, e = rnd(0, q, (cnt, k, l, 256)), rnd(-5, 6, (cnt, l, 256)), rnd(-8, 9, (cnt, k, 256))
            yield ("matvec q=%d k=%d l=%d" % (q, k, l), q, cnt, 4 * 256 * (k * l + l + 2 * k), e,
                   lambda o, pm=pm, A=A, s=s, k=k, l=l: pm.matvec(o, A, s, k, l),
                   lambda o, pm=pm, A=A, s=s, e=e, k=k, l=l: pm.matvec_add(o, A, s, e, k, l))
            A0 = A[0].contiguous()
            del A
            yield ("matvec shared q=%d k=%d l=%d" % (q, k, l), q, cnt, 4 * 256 * (l + 2 * k), e,
                   lambda o, pm=pm, A0=A0, s=s, k=k, l=l: pm.matvec_shared(o, A0, s, k, l),
                   lambda o, pm=pm, A0=A0, s=s, e=e, k=k, l=l: pm.matvec_shared_add(o, A0, s, e, k, l))

    def timed(fn):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(args.calls):
            fn()
        t1.record()
        t1.synchronize()
        return t0.elapsed_time(t1) / 1e3 / args.calls

    result = {"card": card(), "rows": args.rows, "rounds": args.rounds, "calls_per_round": args.calls, "shapes": []}
    for name, q, items, nbytes, e, sib, add in shapes():
        out_f, out_s = torch.empty_like(e), torch.empty_like(e)
        fused = lambda: add(out_f)                                                       # noqa: E731
        alone = lambda: sib(out_s)                                                       # noqa: E731
        def composed():
            sib(out_s)
            torch.remainder(out_s + e, q, out=out_s)
        for fn in (fused, alone, composed):                   # warm-up: modules, the allocator, the scratch pools
            fn()
        torch.cuda.synchronize()
        same = bool(torch.equal(out_f, out_s))                # out_s holds the composition's result here
        times = {"fused": [], "sibling": [], "composition": []}
        for _ in range(args.rounds):
            times["fused"].append(timed(fused))
            times["sibling"].append(timed(alone))
            times["composition"].append(timed(composed))
        rec = {"shape": name, "items": items, "bytes_per_item": nbytes, "outputs_equal": same}
        for key, ts in times.items():
            rates = sorted(items / t for t in ts)
            rec[key] = {"median_per_s": rates[len(rates) // 2], "min_per_s": rates[0], "max_per_s": rates[-1]}
        rec["fused_hbm_fraction"] = rec["fused"]["median_per_s"] * nbytes / HBM
        rec["fused_over_sibling"] = rec["fused"]["median_per_s"] / rec["sibling"]["median_per_s"]
        rec["fused_over_composition"] = rec["fused"]["median_per_s"] / rec["composition"]["median_per_s"]
        result["shapes"].append(rec)
        print("%-32s fused %.3e/s (%.2f of HBM)  sibling %.3e/s  composition %.3e/s  fused/sibling %.3f  "
              "fused/composition %.2f  equal %s" % (name, rec["fused"]["median_per_s"], rec["fused_hbm_fraction"],
                                                    rec["sibling"]["median_per_s"], rec["composition"]["median_per_s"],
                                                    rec["fused_over_sibling"], rec["fused_over_composition"], same),
              flush=True)
        del out_f, out_s, e, sib, add
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("card:", result["card"])
    assert all(r["outputs_equal"] for r in result["shapes"]), "fused and composed outputs differ"


if __name__ == "__main__":
    main()
