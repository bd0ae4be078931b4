"""Does the reference link against libscgpu.so once its own hot-path objects are removed?  (INTEGRATION.md 1)

Runs tools/link_check.sh where the reference sources are available (REF=<their directory>): every reference object
outside the replaced set -- all schemes, module_lwe.c, mw_bootstrap.c, the rest of arith / sampling / crypto -- is
compiled and linked with -lscgpu; no symbol they need from the replaced objects may be missing, and the link may
not leave any prng_* / sampler / NTT symbol unresolved.  On boxes without the sources the committed output of the
same script (profiles/link_check_r2.txt) is checked against the library's export list."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEEDED = ("barrett_init create_sampler destroy_sampler get_bootstrap_sample get_sample get_vector_32 init_reduce prng_32 "
          "prng_64 prng_8 prng_bit prng_create prng_destroy prng_double prng_get_type prng_init prng_mem prng_set_entropy "
          "prng_var set_discard").split()
# the rest of prng.h:38-100 and sampling.h:88-110 (callers: src/safecrypto.c, which needs configure's generated headers)
ALSO = ("utils_arith_ntt ntt_table prng_reset prng_128 prng_float prng_double prng_16 prng_get_csprng_bytes "
        "prng_get_out_bytes prng_set_entropy_callback get_vector_16 roots_of_unity_s16 roots_of_unity_s32").split()


def exported():
    import libsafecrypto_b200 as sc
    if not os.path.exists(sc.lib_path()):
        import __graft_entry__ as ge
        ge.build()
    out = subprocess.run(["nm", "-D", "--defined-only", sc.lib_path()], capture_output=True, text=True, check=True).stdout
    return {line.split()[-1] for line in out.splitlines() if line.strip()}


def test_committed_link_surface_is_exported():
    text = open(os.path.join(ROOT, "profiles", "link_check_r2.txt")).read()
    m = re.search(r"symbols the kept objects need from the replaced ones:\n(.*)\n", text)
    needed = m.group(1).split()
    assert sorted(needed) == sorted(NEEDED)
    exp = exported()
    for name in needed + ALSO:
        assert name in exp, name
    assert re.search(r"missing from libscgpu.so:\n\s*\n", text)


# the reference's source tree, named by REF as for oracle/Makefile and tools/link_check.sh
REF = os.environ.get("REF", "")


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))), reason="reference sources not present (set REF)")
def test_reference_links_against_libscgpu():
    res = subprocess.run(["sh", os.path.join(ROOT, "tools", "link_check.sh")], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    out = res.stdout
    assert re.search(r"missing from libscgpu.so:\n\s*\n", out), out[-2000:]
    unresolved = re.findall(r"`([A-Za-z_0-9]+)'", out.split("link: gcc")[1])
    bad = [s for s in unresolved if s.startswith(("prng_", "ntt", "get_vector", "get_sample", "get_bootstrap", "create_sampler", "destroy_sampler", "set_discard",
                                                   "init_reduce", "barrett_init", "utils_arith", "roots_of_unity"))]
    assert not bad, bad
    assert "kept objects: 10" in out            # 100+ reference objects took part in the link
