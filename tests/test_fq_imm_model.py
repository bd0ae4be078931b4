"""CPU check of the pass-0 products with the entries as instruction immediates (fq_arith.cuh: make_imm, mul_imm;
fq_host.h: analyse32_bm_imm): tools/fq_model.cpp runs the base-multiplication schedule with pass 0 through mul_imm
against a schoolbook product.  The analysis must accept the reference's (12289, 512) table and refuse a modulus whose
base-multiplication bounds do not hold."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_immediate_pass0_model_and_analysis(tmp_path):
    exe = str(tmp_path / "fq_model")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(ROOT, "libsafecrypto_b200", "csrc"),
                           os.path.join(ROOT, "tools", "fq_model.cpp"), "-o", exe])
    out = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout[-2000:]
    verdict, current = {}, None
    for line in out.stdout.splitlines():
        if line.startswith("q="):
            current = tuple(int(f.split("=")[1].rstrip(":")) for f in line.split()[:2])
        elif "pass 0 with immediate entries" in line:
            verdict[current] = "accepted" in line
    assert verdict[(12289, 512)] is True
    assert verdict[(18433, 1024)] is False
    assert verdict[(40961, 512)] is False
