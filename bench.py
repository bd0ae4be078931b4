#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native lattice hot path.

Workload (BASELINE.json configs[1]): batched negacyclic polynomial multiplication, n = 512,
q = 12289, 2^20 independent operand pairs per GPU, synthetic uniform coefficients.  One "step" is
one pass of the fused polymul kernel over the whole batch.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

N > 1 is launched by the driver under torch.distributed.run (one rank per GPU).  The batch shards by
polynomial index with no data-path collective (weak scaling: 2^20 pairs per GPU); NCCL is used only for
the barrier and the max-over-ranks of the device time.

Prints ONE JSON line.  `value` = polymuls/s with operands resident in HBM (CUDA events on the launching
stream); `e2e` = the same metric through scgpu_polymul_batch_host() with pinned HOST buffers, H2D and
D2H inside the timed region (that leg runs max(3, min(K, 10)) steps, recorded as e2e.steps; `--steps K`
sets the device-resident leg's count); `roofline` = algorithmic bytes (12 n per product) / kernel time against
the measured HBM copy bandwidth; `cpu_baseline` = the reference's own C code (oracle/_ref) on the
host cores of this box.  `--impl reference` times that CPU path alone.  `--dump-outputs DIR` writes a fixed,
seeded sample of 2^14 rows of the last timed step's product (rank 0) to DIR/polymul_out.npy as float32; the
operands are seeded, so two builds given the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_COEF, Q = 512, 12289
BATCH = 1 << 20                 # polynomial pairs per GPU per step (device-resident leg)
E2E_BATCH = 1 << 18             # pairs per GPU per step through the host-buffer C-ABI call
METRIC = "ntt_polymul_per_s_n512_q12289"
UNIT = "polymul/s"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def instr_counts():
    """warp-instructions per unit of the hot kernels, from the committed ncu captures (profiles/instr_counts_r2.json,
    written by tools/instr_counts.py from `ncu --set full` reports; instruction counts do not depend on clocks)."""
    path = os.path.join(ROOT, "profiles", "instr_counts_r2.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)
    return {}


def issue_peak(sm_count, sm_mhz):
    """Hardware warp-instruction issue rate: SMs x 4 schedulers x 1 warp-instruction per clock."""
    return sm_count * 4 * sm_mhz * 1e6


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_reference_run(count, threads=0, variant=None, repeats=1):
    """Time the reference's CPU polymul (fwd, fwd, pointwise, inv per pair) on `count` pairs.
    threads = 0 means every host thread this process may run on (explicit, so that torchrun's
    OMP_NUM_THREADS=1 does not turn the baseline into a single-core number)."""
    import _oracle as O
    if threads == 0:
        threads = host_threads()
    if O.ref_available():
        chk, kind = O.ref(), "reference"
        variant = O.AVX if variant is None else variant        # what every scheme selects on an AVX2 host (bliss_b.c:273-277)
    else:
        chk, kind = O.port(), "port"
        variant = O.FP if variant is None else variant
    w, r = O.tables(Q, N_COEF, 16)
    rng = np.random.default_rng(1)
    a = rng.integers(0, Q, size=(count, N_COEF)).astype(np.int32)
    b = rng.integers(0, Q, size=(count, N_COEF)).astype(np.int32)
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        chk.ntt_batch(variant, O.OP_POLYMUL, N_COEF, Q, 16, a, b, w, r, threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    cores = threads
    return count / best, cores, kind, O.VARIANT_NAMES[variant], best


def run_reference_arm(args, rank):
    if rank != 0:
        return
    # bounded sample per step, sized from a short calibration so the whole run stays within minutes
    rate, cores, kind, vname, _ = cpu_reference_run(1 << 14)
    per_step = int(min(1 << 20, max(1 << 14, rate * 1.5)))       # ~1.5 s of CPU work per step
    per_step = 1 << (per_step.bit_length() - 1)
    for _ in range(args.warmup):
        cpu_reference_run(per_step)
    t_total = 0.0
    for _ in range(args.steps):
        _, _, _, _, dt = cpu_reference_run(per_step)
        t_total += dt
    value = per_step * args.steps / t_total
    sample = "%d polymul pairs per step (fwd,fwd,pointwise,inv; variant %s), OpenMP static over %d host threads" % (per_step, vname, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": "batched NTT polymul n=512 q=12289 (BLISS-B / Falcon-512 shape), CPU reference on a bounded sample",
                   "n": N_COEF, "q": Q, "pairs_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


_JSON_FD = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def bind_to_gpu_numa_node(index):
    """Best effort: run this rank (and first-touch its pinned staging buffers) on the CPUs NVML reports as local
    to the GPU, so that the host side of the end-to-end leg does not cross sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
        return len(cpus)
    except Exception:
        return 0


DUMP_ROWS = 1 << 14             # 2^14 of the 2^20 products x 512 coefficients in float32 = 32 MiB


def dump_outputs(path, out):
    """What the timed path returned in its last step, for comparing two builds output for output: the same seeded
    sample of rows of `out` (rank 0's batch) on every run.  Residues are below 2^24, so float32 holds them exactly."""
    import torch
    rows = np.sort(np.random.default_rng(20261020).choice(out.shape[0], size=min(DUMP_ROWS, out.shape[0]), replace=False))
    sample = out[torch.from_numpy(rows).to(out.device)].cpu().numpy().astype(np.float32)
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "polymul_out.npy"), sample)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write a fixed sample of the last timed step's polymul output to DIR/polymul_out.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        # the reference arm sizes its sample from a timing calibration, so its inputs differ from run to run
        ap.error("--dump-outputs applies to --impl ours only")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # The contract is ONE JSON line on stdout.  Libraries may print banners there from C code (NCCL's version
    # line did on an 8-GPU box), so everything else this process writes to fd 1 goes to stderr and the JSON line
    # is written to the saved descriptor at the end.
    sys.stdout.flush()
    global _JSON_FD
    _JSON_FD = os.dup(1)
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    import libsafecrypto_b200 as sc
    import _oracle as O

    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback)"
    if world > 1:
        bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    w, r = O.tables(Q, N_COEF, 16)        # twiddle tables (host set-up; validated against the reference's generated ones)
    plan = sc.NttPlan(N_COEF, Q, sc.REFERENCE, w, r, device=local_rank)
    # the operands are canonical residues (as at every call site of the reference): the plan says so and the fused
    # product skips its per-coefficient range vote; the default path (exact for ANY SINT32) is timed below as well
    plan.set_flags(sc.PLAN_INPUTS_IN_RANGE)
    plan_checked = sc.NttPlan(N_COEF, Q, sc.REFERENCE, w, r, device=local_rank)
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    a = torch.randint(0, Q, (BATCH, N_COEF), dtype=torch.int32, device=dev, generator=g)
    b = torch.randint(0, Q, (BATCH, N_COEF), dtype=torch.int32, device=dev, generator=g)
    out = torch.empty_like(a)

    # ---- device-resident leg ---------------------------------------------------------------------------
    # clocks / throttle reasons are sampled from the first warm-up step to the end of the end-to-end leg
    # (the device-resident timed region alone lasts tens of milliseconds, shorter than one nvidia-smi poll)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        plan.polymul(out, a, b)
    barrier()
    launches0 = sc.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = []
    barrier()
    ev0.record()
    evs = []
    for _ in range(args.steps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        plan.polymul(out, a, b)
        e.record()
        evs.append((s, e))
    ev1.record()
    barrier()
    launches = sc.launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    elapsed_ms = ev0.elapsed_time(ev1)
    kernel_ms = [s.elapsed_time(e) for s, e in evs]
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * BATCH / (ms_per_step * 1e-3)

    # the WHOLE timed output against the checker (rank 0): the compiled reference's own fwd, fwd, pointwise, inv on
    # all host threads when oracle/_ref is present (about 2 s for 2^20 pairs), else the port; other ranks spot-check
    parity = None
    if rank == 0:
        chk, kind = (O.ref(), "reference") if O.ref_available() else (O.port(), "port")
        t0 = time.perf_counter()
        exp = chk.ntt_batch(O.REFERENCE, O.OP_POLYMUL, N_COEF, Q, 16, a.cpu().numpy(), b.cpu().numpy(), w, r, threads=host_threads())
        got = out.cpu().numpy()
        assert np.array_equal(got, exp), "polymul output differs from the oracle"
        parity = {"rows_compared": int(BATCH), "checker": kind, "seconds": time.perf_counter() - t0, "equal": True}
        del exp, got
    else:
        sl = slice(4321, 4321 + 16)
        exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, N_COEF, Q, 16, a[sl].cpu().numpy(), b[sl].cpu().numpy(), w, r)
        assert np.array_equal(out[sl].cpu().numpy(), exp), "polymul output differs from the oracle"

    # ---- roofline of the dominant (only) kernel ------------------------------------------------------------
    peak, peak_src = measured_peaks()
    k_ms = float(np.mean(kernel_ms))
    alg_bytes = 12 * N_COEF * BATCH                     # read a, b (4n each) + write out (4n) per product
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": None, "peak_source": peak_src, "kernel": "k_polymul_w32<ArFq,9,POLYMUL,TMA,BM=1,CHK=0>",
                "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg_bytes}
    prof = os.path.join(ROOT, "profiles", "polymul_traffic.json")
    if os.path.exists(prof):
        with open(prof) as f:
            roofline["traffic"] = json.load(f).get("dram_bytes_per_launch")
    int_roof = None
    props = torch.cuda.get_device_properties(dev)
    sm_count = props.multi_processor_count
    counts = instr_counts()
    if rank == 0:
        # Issue roofline: the kernel is bound by instruction issue, not HBM (DESIGN.md 4.1).  Denominator = the
        # hardware's issue rate, SMs x 4 schedulers x SM clock (the maximum clock: what the part can do); numerator =
        # warp-instructions per product (ncu count of the committed capture of this kernel) x products / s.  A better
        # butterfly therefore shows up as fewer instructions per product at the same fraction, i.e. as throughput.
        smi = sampler.summary() if sampler.rows else {}
        sm_mhz = smi.get("sm_max_mhz") or props.clock_rate / 1e3
        peak_issue = issue_peak(sm_count, sm_mhz)
        ckey = "k_polymul_w32_n512_inrange" if "k_polymul_w32_n512_inrange" in counts else "k_polymul_w32_n512"
        wipp = counts.get(ckey, {}).get("per_unit")
        # arithmetic floor of the schedule: 3 transforms x (log n - 2) stages x n/2 butterflies x 5 instructions, plus
        # n/4 base multiplications x 60 (DESIGN.md 4.1), per warp-instruction of 32 lanes
        arith = (3 * (N_COEF // 2) * 7 * 5 + (N_COEF // 4) * 60) / 32.0
        int_roof = {"bound": "issue", "unit": "warp-instructions/s", "peak": peak_issue, "sm_count": sm_count, "sm_mhz": sm_mhz,
                    "warp_instr_per_product": wipp, "arithmetic_warp_instr_per_product": arith,
                    "source": counts.get(ckey, {}).get("source"), "counted_kernel": ckey,
                    "peak_source": "SMs x 4 schedulers x max SM clock"}
        if wipp:
            ach = wipp * BATCH / (k_ms * 1e-3)
            int_roof.update({"achieved": ach, "frac": ach / peak_issue, "arithmetic_instr_frac": arith / wipp})
    def timed(fn, reps=10):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        s0, e0 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(reps):
            fn()
        e0.record()
        torch.cuda.synchronize()
        return s0.elapsed_time(e0) / reps * 1e-3

    shapes = None
    checked_path = None
    if rank == 0:
        # the default path of the same kernel: range vote on every coefficient, exact for any SINT32 operand
        tc = timed(lambda: plan_checked.polymul(out, a, b))
        checked_path = {"value": BATCH / tc, "unit": UNIT, "hbm_frac": alg_bytes / tc / 1e9 / peak,
                        "kernel": "k_polymul_w32<ArFq,9,POLYMUL,TMA,BM=1,CHK=1>",
                        "note": "scgpu_polymul_batch without SCGPU_PLAN_INPUTS_IN_RANGE (any SINT32 input exact), same operands, same output"}
        shapes = {}

        def put(name, units, secs, bytes_per_unit, unit, ckey=None):
            shapes[name] = {"per_s": units / secs, "unit": unit + "/s", "units": units,
                            "hbm_frac": bytes_per_unit * units / secs / 1e9 / peak}
            # the INT side of the roofline for the same leg: warp-instructions per unit (ncu count of the committed probe
            # of this kernel, profiles/instr_counts_r2.json) x units / s against the hardware issue rate; where the capture
            # shows one pipe busier than the issue slots (IMAD / IMAD.HI on the fma-heavy pipe of the 23-bit moduli) that
            # pipe's utilisation under ncu is quoted beside it
            c = counts.get(ckey) if ckey else None
            if c and c.get("per_unit"):
                shapes[name]["issue_frac"] = c["per_unit"] * units / secs / peak_issue
                shapes[name]["warp_instr_per_unit"] = c["per_unit"]
                if c.get("fmaheavy_pipe_pct"):
                    shapes[name]["fmaheavy_pipe_pct_under_ncu"] = c["fmaheavy_pipe_pct"]

        for (qq, nn) in ((12289, 1024), (7681, 256)):
            ww, rr = O.tables(qq, nn, 16)
            pl = sc.NttPlan(nn, qq, sc.REFERENCE, ww, rr, device=local_rank)
            bb = (1 << 30) // (4 * nn)
            xa = torch.randint(0, qq, (bb, nn), dtype=torch.int32, device=dev, generator=g)
            xb = torch.randint(0, qq, (bb, nn), dtype=torch.int32, device=dev, generator=g)
            xo = torch.empty_like(xa)
            put("polymul_n%d_q%d" % (nn, qq), bb, timed(lambda: pl.polymul(xo, xa, xb)), 12 * nn, "polymul")
            pl.set_flags(sc.PLAN_INPUTS_IN_RANGE)
            put("polymul_n%d_q%d_inputs_in_range" % (nn, qq), bb, timed(lambda: pl.polymul(xo, xa, xb)), 12 * nn, "polymul",
                ckey="k_polymul_w32_n1024_inrange" if nn == 1024 else "k_polymul_w32_n256_q7681_inrange")
            pl.set_flags(0)
            if nn == 256:
                # Kyber module product t = A s, k = l = 3 (module_lwe.c:669-748), A in the NTT domain: 4 n (k^2 + 2 k) bytes
                k = 3
                inst = 1 << 17
                A = torch.randint(0, qq, (inst, k * k, nn), dtype=torch.int32, device=dev, generator=g)
                sv = torch.randint(-4, 5, (inst, k, nn), dtype=torch.int32, device=dev, generator=g)
                to = torch.empty((inst, k, nn), dtype=torch.int32, device=dev)
                put("kyber_matvec_k3_n256_q7681", inst, timed(lambda: pl.matvec(to, A, sv, k, k)), 4 * nn * (k * k + 2 * k), "instance")
                pl.set_flags(sc.PLAN_INPUTS_IN_RANGE)
                put("kyber_matvec_k3_n256_q7681_inputs_in_range", inst, timed(lambda: pl.matvec(to, A, sv, k, k)), 4 * nn * (k * k + 2 * k), "instance",
                    ckey="k_matvec16_w32_kyber_k3_inrange")
                pl.set_flags(0)
                # the same product with the matrix sampled on the device from a 32-byte seed per instance
                # (create_rand_product_16_csprng): 4 n (l + k) + 32 bytes of HBM per instance, generator-bound
                sd = torch.randint(0, 256, (inst, 32), dtype=torch.uint8, device=dev, generator=g)
                for pname, prng in (("chacha20", sc.PRNG_CHACHA), ("aes_ctr_drbg", sc.PRNG_AES_CTR_DRBG)):
                    put("kyber_rand_product_k3_%s" % pname, inst, timed(lambda: pl.rand_product(to, sv, sd, prng, 13, k, k), reps=5),
                        4 * nn * 2 * k + 32, "instance")
                del A, sv, to, sd
            del xa, xb, xo, pl
        # BLISS sign / verify core: v = INTT(NTT(t) o key), one shared SINT16 key (bliss_b.c:1378-1384): 8 n bytes
        key = torch.randint(0, Q, (N_COEF,), dtype=torch.int32, device=dev, generator=g).to(torch.int16)
        put("bliss_key_product_n512_q12289", BATCH, timed(lambda: plan_checked.mul_key(out, a, key)), 8 * N_COEF, "product")
        put("bliss_key_product_n512_q12289_inputs_in_range", BATCH, timed(lambda: plan.mul_key(out, a, key)), 8 * N_COEF, "product",
            ckey="k_polymul_w32_key16_n512_inrange")
        # single transforms with canonical output (normalize_32 o fwd_ntt, inv_ntt), n = 512: 8 n bytes each
        put("fwd_ntt_canonical_n512_q12289", BATCH, timed(lambda: plan.ntt_canonical(out, a)), 8 * N_COEF, "ntt", ckey="k_ntt_w32_fwd_n512_inrange")
        put("inv_ntt_canonical_n512_q12289", BATCH, timed(lambda: plan.ntt_canonical(out, a, inverse=True)), 8 * N_COEF, "ntt", ckey="k_ntt_w32_inv_n512_inrange")
        # the members the drop-in table calls: the variant's own lazily reduced representative, bit for bit
        for vv, vname in ((sc.REFERENCE, "reference"), (sc.BARRETT, "barrett"), (sc.AVX, "avx")):
            pe = sc.NttPlan(N_COEF, Q, vv, w, r, device=local_rank)
            put("exact_fwd_ntt_32_16_n512_%s" % vname, BATCH, timed(lambda: pe.batch(sc.OP_FWD, out, a)), 8 * N_COEF, "ntt", ckey="k_exact_w32_fwd_n512_%s" % vname)
            put("exact_inv_ntt_32_16_n512_%s" % vname, BATCH, timed(lambda: pe.batch(sc.OP_INV, out, a)), 8 * N_COEF, "ntt", ckey="k_exact_w32_inv_n512_%s" % vname)
            del pe
        # Dilithium q = 8380417, n = 256 (32-bit tables): polymul and the k = 5, l = 4 module product
        qq, nn = 8380417, 256
        ww, rr = O.tables(qq, nn, 32)
        pl = sc.NttPlan(nn, qq, sc.REFERENCE, ww, rr, device=local_rank)
        bb = 1 << 20
        xa = torch.randint(0, qq, (bb, nn), dtype=torch.int32, device=dev, generator=g)
        xb = torch.randint(0, qq, (bb, nn), dtype=torch.int32, device=dev, generator=g)
        xo = torch.empty_like(xa)
        put("polymul_n256_q8380417", bb, timed(lambda: pl.polymul(xo, xa, xb)), 12 * nn, "polymul")
        pl.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        put("polymul_n256_q8380417_inputs_in_range", bb, timed(lambda: pl.polymul(xo, xa, xb)), 12 * nn, "polymul",
            ckey="k_polymul_w32_n256_q8380417_inrange")
        pl.set_flags(0)
        del xa, xb, xo
        inst = 1 << 15
        A = torch.randint(0, qq, (inst, 20, nn), dtype=torch.int32, device=dev, generator=g)
        sv = torch.randint(-2, 3, (inst, 4, nn), dtype=torch.int32, device=dev, generator=g)
        to = torch.empty((inst, 5, nn), dtype=torch.int32, device=dev)
        put("dilithium_matvec_k5_l4_n256", inst, timed(lambda: pl.matvec(to, A, sv, 5, 4)), 4 * nn * (20 + 4 + 5), "instance")
        pl.set_flags(sc.PLAN_INPUTS_IN_RANGE)
        put("dilithium_matvec_k5_l4_n256_inputs_in_range", inst, timed(lambda: pl.matvec(to, A, sv, 5, 4)), 4 * nn * (20 + 4 + 5), "instance",
            ckey="k_matvec_w32_dilithium_k5_l4_inrange")
        del A, sv, to, pl

    # ---- end-to-end leg: host buffers through the C-ABI ----------------------------------------------------
    ha = torch.randint(0, Q, (E2E_BATCH, N_COEF), dtype=torch.int32).pin_memory()
    hb = torch.randint(0, Q, (E2E_BATCH, N_COEF), dtype=torch.int32).pin_memory()
    ho = torch.empty((E2E_BATCH, N_COEF), dtype=torch.int32).pin_memory()
    for _ in range(2):
        plan.polymul_host(ho, ha, hb)
    barrier()
    e2e_steps = max(3, min(args.steps, 10))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        plan.polymul_host(ho, ha, hb)                    # blocks until the result is back in host memory
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * E2E_BATCH * e2e_steps / e2e_s
    sampler.stop_flag.set()
    sampler.join()
    exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, N_COEF, Q, 16, ha[:8].numpy(), hb[:8].numpy(), w, r)
    assert np.array_equal(ho[:8].numpy(), exp), "host-path output differs from the oracle"
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * 4 * N_COEF * E2E_BATCH,
           "d2h_bytes_per_step": 4 * N_COEF * E2E_BATCH, "pairs_per_step": E2E_BATCH, "steps": e2e_steps,
           "api": "scgpu_polymul_batch_host (pinned host buffers, chunked 3-stream H2D/kernel/D2H pipeline)"}

    # ---- composed end-to-end leg: the BLISS-B sign core (bliss_b.c:1372-1384) through the C-ABI, seeds in, v out ------
    # t = get_vector_32(sigma 215) on the device from a 40-byte seed per signature, v = INTT(NTT(t) o a) with the public
    # key a resident on the device; only the seeds cross the bus on the way in (40 B) and v on the way out (4 n B).
    sign_core = None
    if rank == 0:
        gps = sc.GaussPlan(sc.SAMPLER_CDF, 64, 0, 13.42, 215.0, device=local_rank)
        nsig = 1 << 18
        chunk = 1 << 16
        hseed = torch.randint(0, 256, (nsig, 40), dtype=torch.uint8).pin_memory()
        hv = torch.empty((nsig, N_COEF), dtype=torch.int32).pin_memory()
        keyd = torch.randint(0, Q, (N_COEF,), dtype=torch.int32, device=dev, generator=g).to(torch.int16)
        streams = [torch.cuda.Stream(device=dev) for _ in range(3)]
        bufs = [(torch.empty((chunk, 40), dtype=torch.uint8, device=dev), torch.empty((chunk, N_COEF), dtype=torch.int32, device=dev),
                 torch.empty((chunk, N_COEF), dtype=torch.int32, device=dev)) for _ in range(3)]

        def sign_pass():
            for ci, off in enumerate(range(0, nsig, chunk)):
                st = streams[ci % 3]
                dseed, dt, dv = bufs[ci % 3]
                with torch.cuda.stream(st):
                    dseed.copy_(hseed[off:off + chunk], non_blocking=True)
                    gps.streams(sc.PRNG_CHACHA, dseed, N_COEF, dt, stream=st)
                    plan.mul_key(dv, dt, keyd, stream=st)
                    hv[off:off + chunk].copy_(dv, non_blocking=True)
            for st in streams:
                st.synchronize()

        sign_pass()
        t0 = time.perf_counter()
        for _ in range(3):
            sign_pass()
        dt_s = (time.perf_counter() - t0) / 3
        # parity of the composition on a few signatures: the port's sampler, then the oracle's triple
        tt = O.port().gauss_streams(O.SAMPLER_CDF, 64, 0, O.PRNG_CHACHA, 13.42, 215.0, hseed[:4].numpy(), N_COEF)
        vv = O.port().ntt_batch(O.REFERENCE, O.OP_TRIPLE16, N_COEF, Q, 16, tt, keyd.cpu().numpy(), w, r)
        assert np.array_equal(hv[:4].numpy(), vv), "sign-core composition differs from the oracle"
        sign_core = {"value": nsig / dt_s, "unit": "sign cores/s (get_vector_32 + fwd_ntt, mul_32_pointwise_16, inv_ntt)", "signatures": nsig,
                     "h2d_bytes_per_step": 40 * nsig, "d2h_bytes_per_step": 4 * N_COEF * nsig,
                     "api": "scgpu_gauss_streams -> scgpu_ntt_mul_key_batch on device buffers, seeds H2D and v D2H inside the timed region"}
        del hseed, hv, bufs

    # ---- strong scaling of ONE host batch from ONE process: the fixed 2^20-pair batch of BASELINE configs[1] split over
    # all GPUs by scgpu_polymul_batch_host_multi (host-side scatter / gather, one thread per device).  Rank 0 drives
    # every device; the other ranks wait on the rendezvous store (a host wait, their GPUs are idle).
    e2e_multi = None
    if world > 1:
        from torch.distributed.distributed_c10d import _get_default_store
        store = _get_default_store()
        barrier()
        if rank == 0:
            from libsafecrypto_b200 import binding as B
            ps = B.NttPlanSet(N_COEF, Q, sc.REFERENCE, w, r, max_devices=world)
            mb = 1 << 20
            ma = torch.randint(0, Q, (mb, N_COEF), dtype=torch.int32).pin_memory()
            mbb = torch.randint(0, Q, (mb, N_COEF), dtype=torch.int32).pin_memory()
            mo = torch.empty((mb, N_COEF), dtype=torch.int32).pin_memory()
            e2e_multi = {"pairs": mb, "api": "scgpu_polymul_batch_host_multi (one process, one thread per device)", "by_devices": {}}
            nd = 1
            while nd <= ps.ndev:
                ps.polymul_host(mo, ma, mbb, ndev=nd)
                t0 = time.perf_counter()
                for _ in range(3):
                    ps.polymul_host(mo, ma, mbb, ndev=nd)
                dt = (time.perf_counter() - t0) / 3
                e2e_multi["by_devices"][str(nd)] = {"polymul_per_s": mb / dt, "seconds": dt}
                nd *= 2
            exp = O.port().ntt_batch(O.REFERENCE, O.OP_POLYMUL, N_COEF, Q, 16, ma[-8:].numpy(), mbb[-8:].numpy(), w, r)
            assert np.array_equal(mo[-8:].numpy(), exp), "multi-device host path differs from the oracle"
            ps.close()
            del ma, mbb, mo
            store.set("scgpu_multi_done", "1")
        else:
            store.wait(["scgpu_multi_done"])
        barrier()

    # ---- secondary metric: Gaussian samples/s (BASELINE config 5 shape), every rank its own streams -------------
    # CDF-64, sigma 215, both generators; "fixed_probe" = the default constant-time table search (the reference's
    # log2(size) probes for every draw), "guided" = the optional guide-bracketed bisection (data-dependent trip count)
    gp = sc.GaussPlan(sc.SAMPLER_CDF, 64, 0, 13.42, 215.0, device=local_rank)
    nstreams, n = 1 << 18, 512
    seeds = torch.randint(0, 256, (nstreams, 40), dtype=torch.uint8, device=dev, generator=g)
    smp = torch.empty((nstreams, n), dtype=torch.int32, device=dev)
    gauss = {}
    smi = sampler.summary() if sampler.rows else {}
    peak_issue = issue_peak(sm_count, smi.get("sm_max_mhz") or props.clock_rate / 1e3)
    for mode, fixed in (("fixed_probe", 1), ("guided", 0)):
        old = sc.lib().scgpu_set_fixed_probe_search(fixed)
        for name, prng in (("aes_ctr_drbg", sc.PRNG_AES_CTR_DRBG), ("chacha20", sc.PRNG_CHACHA)):
            for _ in range(3):
                gp.streams(prng, seeds, n, smp)
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(5):
                gp.streams(prng, seeds, n, smp)
            e.record()
            barrier()
            ms = s.elapsed_time(e)
            if world > 1:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t.item())
            rate = world * 5 * nstreams * n / (ms * 1e-3)
            entry = {"samples_per_s": rate, "hbm_frac": 4 * rate / world / 1e9 / peak}
            key = "k_cdf_%s_%s" % ("aes" if prng == sc.PRNG_AES_CTR_DRBG else "chacha", mode)
            wips = counts.get(key, {}).get("per_unit")
            if wips:
                # issue roofline of the sampler: warp-instructions per sample (ncu, committed capture) x samples/s per GPU
                entry["roofline"] = {"bound": "issue", "warp_instr_per_sample": wips, "achieved": wips * rate / world,
                                     "peak": peak_issue, "frac": wips * rate / world / peak_issue,
                                     "alu_pipe_pct": counts[key].get("alu_pipe_pct"), "source": counts[key].get("source")}
            gauss["cdf64_sigma215_%s_%s" % (name, mode)] = entry
        sc.lib().scgpu_set_fixed_probe_search(old)
    gauss["cdf64_sigma215_aes_ctr_drbg_samples_per_s"] = gauss["cdf64_sigma215_aes_ctr_drbg_fixed_probe"]["samples_per_s"]
    gauss["cdf64_sigma215_chacha20_samples_per_s"] = gauss["cdf64_sigma215_chacha20_fixed_probe"]["samples_per_s"]
    gauss["shape"] = "%d streams x %d samples per GPU on %d GPU(s), CDF-64, sigma 215, tail 13.42; whole-job rate, max over ranks; 4 B of HBM per sample (the roof is instruction issue)" % (nstreams, n, world)
    # spot check against the oracle
    exp = O.port().gauss_streams(O.SAMPLER_CDF, 64, 0, sc.PRNG_CHACHA, 13.42, 215.0, seeds[:4].cpu().numpy(), n)
    assert np.array_equal(smp[:4].cpu().numpy(), exp), "sampler output differs from the oracle"
    # end to end through the C-ABI with HOST buffers: seeds in (40 B per stream), samples out (4 B each), copies inside
    if rank == 0:
        hs = seeds.cpu().pin_memory()
        ho_s = torch.empty((nstreams, n), dtype=torch.int32).pin_memory()
        for name, prng in (("aes_ctr_drbg", sc.PRNG_AES_CTR_DRBG), ("chacha20", sc.PRNG_CHACHA)):
            gp.streams_host(prng, hs, n, ho_s)
            t0 = time.perf_counter()
            for _ in range(3):
                gp.streams_host(prng, hs, n, ho_s)
            dt = (time.perf_counter() - t0) / 3
            gauss["cdf64_sigma215_%s_e2e" % name] = {"samples_per_s": nstreams * n / dt, "h2d_bytes_per_step": 40 * nstreams,
                                                     "d2h_bytes_per_step": 4 * nstreams * n, "api": "scgpu_gauss_streams_host"}
        assert np.array_equal(ho_s[:4].numpy(), exp), "host-path sampler output differs from the oracle"
        del hs, ho_s
    # Knuth-Yao-64 and Bernoulli-64 (the other two samplers north_star names), sigma 215, smaller batches; every rank its
    # own streams, whole-job rate over the slowest rank like the CDF legs
    for sname, sid, ns in (("knuth_yao64", sc.SAMPLER_KNUTH_YAO, 1 << 17), ("bernoulli64", sc.SAMPLER_BERNOULLI, 1 << 17)):
        gpx = sc.GaussPlan(sid, 64, 0, 13.42, 215.0, device=local_rank)
        sx = torch.empty((ns, n), dtype=torch.int32, device=dev)
        for prng_name, prng in (("aes_ctr_drbg", sc.PRNG_AES_CTR_DRBG), ("chacha20", sc.PRNG_CHACHA)):
            barrier()
            secs = timed(lambda: gpx.streams(prng, seeds[:ns], n, sx), reps=3)
            if world > 1:
                t = torch.tensor([secs], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                secs = float(t.item())
            gauss["%s_sigma215_%s_samples_per_s" % (sname, prng_name)] = world * ns * n / secs
        del gpx, sx
    # the reference's own get_vector_32 (CDF-64 through create_sampler) on the host cores, both generators
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        chk, kind = (O.ref(), "reference") if O.ref_available() else (O.port(), "port")
        hseeds = seeds[:1 << 15].cpu().numpy()
        cpu_g = {"kind": kind, "cores": host_threads()}
        for name, prng in (("aes_ctr_drbg", O.PRNG_AES_CTR_DRBG), ("chacha20", O.PRNG_CHACHA)):
            chk.gauss_streams(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, hseeds[:1 << 12], n, threads=host_threads())
            t0 = time.perf_counter()
            chk.gauss_streams(O.SAMPLER_CDF, 64, 0, prng, 13.42, 215.0, hseeds, n, threads=host_threads())
            dt = time.perf_counter() - t0
            cpu_g["cdf64_sigma215_%s_samples_per_s" % name] = hseeds.shape[0] * n / dt
        cpu_g["sample"] = "%d streams x %d samples, create_sampler(CDF, 64-bit) + get_vector_32 per stream, OpenMP over %d host threads" % (hseeds.shape[0], n, host_threads())
        gauss["cpu_baseline"] = cpu_g

    # ---- CPU baseline beside it (rank 0, N = 1 only) ------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        rate, cores, kind, vname, _ = cpu_reference_run(1 << 14)
        count = int(min(1 << 20, max(1 << 14, rate * 12)))         # ~12 s of CPU work
        rate, cores, kind, vname, dt = cpu_reference_run(count)
        rate1, _, _, _, _ = cpu_reference_run(max(1 << 12, count // max(cores, 1)), threads=1)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "%d pairs, variant %s (fwd,fwd,pointwise,inv), %.1f s wall; 1-thread rate %.0f/s" % (count, vname, dt, rate1)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": "batched NTT polymul n=512 q=12289 (BASELINE configs[1]), 2^20 pairs per GPU, fused fwd/fwd/pointwise/inv, canonical output",
                       "n": N_COEF, "q": Q, "pairs_per_gpu": BATCH, "parallelism": "shard by polynomial index, no collective",
                       "cache": "operands 4 GiB + result 2 GiB per step >> 126 MB L2 (no flush needed)",
                       "inputs": "uniform residues in [0, q); plan flag SCGPU_PLAN_INPUTS_IN_RANGE set (no range vote in the kernel); "
                                 "the default any-SINT32-exact path on the same operands is `checked_path`"},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": sampler.summary(), "roofline": roofline,
            "int_roofline": int_roof, "cpu_baseline": cpu, "gaussian": gauss, "checked_path": checked_path, "other_shapes": shapes, "parity": parity, "e2e_multi": e2e_multi, "e2e_bliss_sign_core": sign_core,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
