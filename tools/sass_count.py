"""Static per-region instruction counts of one kernel, from `cuobjdump -sass` (no GPU needed).

Every backward branch closes a loop.  Loops of at least --min-loop instructions are regions; their trip counts per
iteration of the outermost one are given in address order by --trips (smaller loops, the elect / poll loops of the
bulk copies, count once).  The outermost loop's own body, minus its regions, is one more region ("rest", trip 1).  The
sum of count x trips is the static count of one outer iteration; divided by --units (products per warp iteration)
it is per product.  "rest" counts every instruction of the outer body once, including the blocks a warp may branch
around, so it is an upper bound of what is executed; the per-product difference between two builds is exact for
changes that touch only straight-line code.

usage: python tools/sass_count.py [--binary libscgpu.so|obj.o] [--kernel REGEX] [--trips 2,2] [--units 2] [--json]
The defaults are the headline kernel of bench.py: the fused product n = 512 with the base multiplication, bulk-copied
rows, in-range plan (k_polymul_w32<ArFq or ArFqImm, 9, FQ_POLYMUL, TMA, BM, !CHK>), 2 operand passes, 2 sub-chunks,
2 products per warp iteration."""
import argparse
import collections
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADLINE = r"k_polymul_w32INS_\w*?\d(?:ArFq|ArFqImm)ELi9ELi0ELb1ELb1ELb0E"
LINE = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(@!?U?P[T\d]\s+)?([A-Z0-9_.]+)([^;]*);")


def kernels(binary):
    txt = subprocess.run(["cuobjdump", "-sass", binary], capture_output=True, text=True, check=True).stdout
    for chunk in re.split(r"\n\s*Function : ", txt)[1:]:
        name, body = chunk.split("\n", 1)
        ins = []
        for m in LINE.finditer(body):
            op, args = m.group(3), m.group(4)
            tgt = None
            if op.split(".")[0] in ("BRA", "BRX"):
                t = re.search(r"0x([0-9a-f]+)", args)
                tgt = int(t.group(1), 16) if t else None
            ins.append((int(m.group(1), 16), op, tgt))
        yield name.strip(), ins


def regions(ins, min_loop, trips):
    loops = sorted({(tgt, addr) for addr, op, tgt in ins if tgt is not None and tgt <= addr}, key=lambda l: l[0])
    outer = max(loops, key=lambda l: l[1] - l[0])
    size = lambda l: sum(1 for a, _, _ in ins if l[0] <= a <= l[1])
    inner = [l for l in loops if l != outer and outer[0] <= l[0] and l[1] <= outer[1] and size(l) >= min_loop]
    inner = [l for l in inner if not any(o != l and o[0] <= l[0] and l[1] <= o[1] for o in inner)]   # outermost only
    if len(trips) != len(inner):
        sys.exit("%d loops of >= %d instructions inside the outer loop, %d trip counts given" % (len(inner), min_loop, len(trips)))
    out = []
    for (lo, hi), t in zip(inner, trips):
        body = [op for a, op, _ in ins if lo <= a <= hi]
        out.append(("loop 0x%x-0x%x" % (lo, hi), t, body))
    rest = [op for a, op, _ in ins if outer[0] <= a <= outer[1] and not any(lo <= a <= hi for lo, hi in inner)]
    out.append(("rest 0x%x-0x%x" % outer, 1, rest))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--binary", default=os.path.join(ROOT, "libsafecrypto_b200", "libscgpu.so"))
    ap.add_argument("--kernel", default=HEADLINE, help="regular expression over the mangled name (every match is listed)")
    ap.add_argument("--trips", default="2,2", help="trip counts of the inner loops, in address order")
    ap.add_argument("--units", type=float, default=2.0, help="products per outer iteration (polynomials per warp)")
    ap.add_argument("--min-loop", type=int, default=64)
    ap.add_argument("--json", action="store_true")
    args = ap.parse_args()
    trips = [int(t) for t in args.trips.split(",") if t]
    res = []
    for name, ins in kernels(args.binary):
        if not re.search(args.kernel, name):
            continue
        regs = regions(ins, args.min_loop, trips)
        row = {"kernel": name, "regions": []}
        total = total_ldc = 0
        for label, t, body in regs:
            hist = collections.Counter(op.split(".")[0] for op in body)
            ldc = hist["LDC"] + hist["LDCU"]
            row["regions"].append({"region": label, "trips": t, "instructions": len(body), "ldc": ldc,
                                   "top": hist.most_common(8)})
            total += t * len(body)
            total_ldc += t * ldc
        row["per_iteration"] = total
        row["per_product"] = total / args.units
        row["ldc_per_product"] = total_ldc / args.units
        res.append(row)
    if not res:
        sys.exit("no kernel matches %r" % args.kernel)
    if args.json:
        print(json.dumps(res, indent=1))
        return
    for row in res:
        print(row["kernel"])
        for r in row["regions"]:
            print("  %-22s x%d  %5d instructions  %4d LDC/LDCU   %s" % (r["region"], r["trips"], r["instructions"], r["ldc"],
                                                                   ", ".join("%s %d" % kv for kv in r["top"])))
        print("  per outer iteration %d, per product %.1f (of which LDC/LDCU %.1f)" %
              (row["per_iteration"], row["per_product"], row["ldc_per_product"]))


if __name__ == "__main__":
    main()
