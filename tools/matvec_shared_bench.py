"""Module products under one key: per-instance matrices against one shared matrix, on one GPU.

For each shape (Kyber k = 2 / 3 / 4 at q = 7681, Dilithium (5, 4) and (6, 5) at q = 8380417) and each plan (default and
SCGPU_PLAN_INPUTS_IN_RANGE), two pairs are timed with CUDA events, the old and the new call alternating in the same run:
  * matvec (A replicated to [count][k][l][n]) against matvec_shared (A [k][l][n]);
  * rand_product (the seed repeated per instance) against rand_product_shared (one seed), ChaCha20 and AES-CTR-DRBG.
Batches are 2^20 instances for Kyber and 2^19 for Dilithium, so s and t alone are far larger than the 126 MB L2.  Bytes
are algorithmic: 4 n (k l + l + k) per instance for the per-instance product, 4 n (l + k) per instance plus the matrix
once for the shared one; the HBM fraction is against 6550 GB/s.  At the timed size the whole output of each shared call
is compared with its per-instance twin.

usage: python tools/matvec_shared_bench.py --out DIR [--reps R]     (writes DIR/matvec_shared.json)
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import libsafecrypto_b200 as sc  # noqa: E402
import _oracle as O  # noqa: E402

HBM_GBS = 6550.0
N = 256
SHAPES = [("kyber2", 7681, 16, 13, 2, 2, 1 << 20), ("kyber3", 7681, 16, 13, 3, 3, 1 << 20), ("kyber4", 7681, 16, 13, 4, 4, 1 << 20),
          ("dilithium54", 8380417, 32, 23, 5, 4, 1 << 19), ("dilithium65", 8380417, 32, 23, 6, 5, 1 << 19)]
DEV = torch.device("cuda", 0)


def device_info():
    info = {"device": torch.cuda.get_device_name(0), "sm_count": torch.cuda.get_device_properties(0).multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def alternate(fns, reps, warmup):
    """Median seconds per call of each function, the functions interleaved call by call."""
    for _ in range(warmup):
        for f in fns:
            f()
    torch.cuda.synchronize()
    times = [[] for _ in fns]
    for _ in range(reps):
        for i, f in enumerate(fns):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            f()
            e.record()
            e.synchronize()
            times[i].append(s.elapsed_time(e) * 1e-3)
    return [statistics.median(t) for t in times], [min(t) for t in times]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("matvec_shared_bench: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    g = torch.Generator(device=DEV).manual_seed(2024)
    res = {"info": device_info(), "hbm_gbs_reference": HBM_GBS, "reps": args.reps, "results": []}
    all_equal = True
    for name, q, tw, q_bits, k, l, count in SHAPES:
        w, r = O.tables(q, N, tw)
        for flag in (0, sc.PLAN_INPUTS_IN_RANGE):
            p = sc.NttPlan(N, q, sc.REFERENCE, w, r)
            if flag:
                p.set_flags(flag)
            A = torch.randint(0, q, (k, l, N), dtype=torch.int32, device=DEV, generator=g)
            s = torch.randint(-5, 6, (count, l, N), dtype=torch.int32, device=DEV, generator=g)
            Arep = A.unsqueeze(0).expand(count, k, l, N).contiguous()
            o_old = torch.empty((count, k, N), dtype=torch.int32, device=DEV)
            o_new = torch.empty_like(o_old)
            (t_old, t_new), (m_old, m_new) = alternate([lambda: p.matvec(o_old, Arep, s, k, l),
                                                        lambda: p.matvec_shared(o_new, A, s, k, l)], args.reps, args.warmup)
            torch.cuda.synchronize()
            eq = bool(torch.equal(o_old, o_new))
            all_equal &= eq
            b_old = 4 * N * (k * l + l + k) * count
            b_new = 4 * N * (l + k) * count + 4 * N * k * l
            row = {"shape": name, "q": q, "k": k, "l": l, "count": count, "plan": "in_range" if flag else "default",
                   "pair": "matvec", "equal": eq,
                   "per_instance": {"s": t_old, "min_s": m_old, "inst_per_s": count / t_old, "bytes": b_old,
                                    "hbm_fraction": b_old / t_old / 1e9 / HBM_GBS},
                   "shared": {"s": t_new, "min_s": m_new, "inst_per_s": count / t_new, "bytes": b_new,
                              "hbm_fraction": b_new / t_new / 1e9 / HBM_GBS},
                   "speedup": t_old / t_new}
            res["results"].append(row)
            print(json.dumps(row), flush=True)
            del Arep
            for pname, prng in (("chacha20", sc.PRNG_CHACHA), ("aes_ctr_drbg", sc.PRNG_AES_CTR_DRBG)):
                seed = torch.randint(0, 256, (32,), dtype=torch.uint8, device=DEV, generator=g)
                seeds = seed.unsqueeze(0).expand(count, 32).contiguous()
                (t_old, t_new), (m_old, m_new) = alternate([lambda: p.rand_product(o_old, s, seeds, prng, q_bits, k, l),
                                                            lambda: p.rand_product_shared(o_new, s, seed, prng, q_bits, k, l)],
                                                           args.reps, args.warmup)
                torch.cuda.synchronize()
                eq = bool(torch.equal(o_old, o_new))
                all_equal &= eq
                row = {"shape": name, "q": q, "k": k, "l": l, "count": count, "plan": "in_range" if flag else "default",
                       "pair": "rand_product_" + pname, "equal": eq,
                       "per_seed": {"s": t_old, "min_s": m_old, "inst_per_s": count / t_old},
                       "shared_seed": {"s": t_new, "min_s": m_new, "inst_per_s": count / t_new,
                                       "hbm_fraction": b_new / t_new / 1e9 / HBM_GBS},
                       "speedup": t_old / t_new}
                res["results"].append(row)
                print(json.dumps(row), flush=True)
                del seeds
            del s, o_old, o_new
            p.close()
            torch.cuda.empty_cache()
    res["all_equal"] = all_equal
    with open(os.path.join(args.out, "matvec_shared.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"info": res["info"], "all_equal": all_equal}))
    if not all_equal:
        sys.exit("matvec_shared_bench: a shared result differs from its per-instance twin")


if __name__ == "__main__":
    main()
