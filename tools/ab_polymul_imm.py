"""A/B of the fused product n = 512, q = 12289 (2^20 pairs, uniform residues, in-range plan as in bench.py): the kernel
with the pass-0 entries compiled in as immediates (ArFqImm, chosen for the reference's table) against the table-driven
kernel, forced by the table of another primitive 2n-th root (same products).  The two alternate `--rounds` times in one
process; each sample is the mean of `--reps` launches between CUDA events.  Outputs are compared in full.
usage: python tools/ab_polymul_imm.py [--rounds 12] [--reps 20] [--out result.json]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import libsafecrypto_b200 as sc  # noqa: E402
import _oracle as O  # noqa: E402

Q, N, B = 12289, 512, 1 << 20


def perturbed_tables():
    w, _ = O.tables(Q, N, 16)
    g = pow(int(w[1]), 3, Q)
    ninv = pow(N, Q - 2, Q)
    wp = [pow(g, i, Q) for i in range(N)]
    return np.array(wp, dtype=np.int16), np.array([(Q - ninv) * x % Q for x in wp], dtype=np.int16)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        return out
    except Exception as e:                               # noqa: BLE001
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=12)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1)
    plans = {}
    for name, (w, r) in (("immediate", O.tables(Q, N, 16)), ("table", perturbed_tables())):
        p = sc.NttPlan(N, Q, sc.REFERENCE, w, r)
        p.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        plans[name] = p
    a = torch.randint(0, Q, (B, N), dtype=torch.int32, device=dev, generator=g)
    b = torch.randint(0, Q, (B, N), dtype=torch.int32, device=dev, generator=g)
    outs = {k: torch.empty((B, N), dtype=torch.int32, device=dev) for k in plans}
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for k, p in plans.items():                           # warm-up of both kernels
        for _ in range(3):
            p.polymul(outs[k], a, b)
    torch.cuda.synchronize()
    rates = {k: [] for k in plans}
    for _ in range(args.rounds):
        for k, p in plans.items():
            s.record()
            for _ in range(args.reps):
                p.polymul(outs[k], a, b)
            e.record()
            e.synchronize()
            rates[k].append(B * args.reps / (s.elapsed_time(e) * 1e-3))
    equal = torch.equal(outs["immediate"], outs["table"])
    res = {"card": card(), "pairs": B, "rounds": args.rounds, "reps": args.reps, "outputs_equal": equal}
    for k, v in rates.items():
        res[k] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v)), "samples": v}
    res["gain_median"] = res["immediate"]["median"] / res["table"]["median"] - 1
    res["spreads_overlap"] = res["immediate"]["min"] <= res["table"]["max"]
    print("card: %s" % res["card"])
    for k in plans:
        print("%-10s median %.4g polymul/s  [min %.4g, max %.4g]" % (k, res[k]["median"], res[k]["min"], res[k]["max"]))
    print("gain of the immediate kernel by median: %+.2f %%, spreads overlap: %s, outputs equal: %s" % (
        100 * res["gain_median"], res["spreads_overlap"], equal))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    sys.exit(0 if equal else 1)


if __name__ == "__main__":
    main()
