"""CPU checks of the drop-in boundary: the C-ABI library builds, loads, and exports every symbol the
headers declare; the product never touches oracle/; without a GPU every entry point fails loudly."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import util

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    names = set()
    for hdr in ("smvp_cuda.h", "smvp_synth.h"):
        text = open(os.path.join(REPO, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names |= set(re.findall(r"\b(smvp_[a-z0-9_]+)\s*\(", text))
    return names


@pytest.fixture(scope="module")
def eng():
    import smvp_toolkit_b200 as e

    if not os.path.exists(e.LIB_PATH):
        import __graft_entry__

        __graft_entry__.build()
    return e


def test_library_exports_every_declared_symbol(eng):
    L = eng.lib()
    decl = declared_symbols()
    assert len(decl) >= 30
    for name in decl:
        assert hasattr(L, name), "libsmvp_cuda.so does not export %s" % name
    assert decl == set(eng.SIGNATURES), "engine.py's ctypes table and the headers disagree"
    out = subprocess.run(["nm", "-D", "--defined-only", eng.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (\w+)", out))
    assert decl <= exported
    # nothing but the C ABI leaks out of the library
    assert all(s.startswith("smvp_") for s in exported), exported - decl


def test_library_is_sm100a_with_tma(eng):
    """The kernels are compiled for sm_100a and the merge-path kernel stages tiles with TMA bulk copies."""
    out = subprocess.run(["cuobjdump", "-lelf", eng.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    sass = subprocess.run(["cuobjdump", "-sass", eng.LIB_PATH], capture_output=True, text=True).stdout
    assert "UBLKCP" in sass  # cp.async.bulk global->shared
    assert "SYNCS" in sass   # mbarrier


def test_hot_kernels_do_not_spill(eng):
    """A register spill in the multiply kernels halves their throughput (measured, profiles/): the build must
    stay spill-free (STACK:0) for every CSR / TJDS multiply kernel.  One deliberate exception, decided by measurement
    (profiles/r02_logs/r02_tjds_sweep5.log): the one-word deterministic TJDS kernel is forced to 32 registers for 8 CTAs per
    SM and keeps ONE 4-byte value on the stack (3.0 - 3.1 ms against 3.85 ms spill-free at 6 CTAs per SM)."""
    out = subprocess.run(["cuobjdump", "-res-usage", eng.LIB_PATH], capture_output=True, text=True).stdout
    lines = out.splitlines()
    seen = 0
    allowed = {"tjds_det_kernelILi4ELb1ELb1ELi8ELi1E": 8}  # <UNROLL 4, skewed, fast split, 8 CTAs/SM, one word>
    for i, ln in enumerate(lines):
        if "Function" in ln and re.search(r"csr_merge_warp_kernel|csr_vector_kernel|tjds_atomic_kernel|tjds_det_kernel", ln):
            usage = lines[i + 1]
            m = re.search(r"STACK:(\d+)", usage)
            limit = max([v for k, v in allowed.items() if k in ln] + [0])
            assert m and int(m.group(1)) <= limit, (ln, usage)
            seen += 1
    assert seen >= 4


def test_no_gpu_means_loud_failure_not_fallback(eng):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    m, n, coo = util.load_sample("pdp08-pg4")
    with pytest.raises(eng.SmvpError) as ei:
        eng.smvp_csr_compute(coo, m, len(coo), 1)
    assert ei.value.code == eng.E_CUDA
    with pytest.raises(eng.SmvpError):
        eng.smvp_tjds_compute(coo, m, n, len(coo), 1)


def _header_fields(struct):
    """field names of a struct typedef in include/smvp_cuda.h, in declaration order"""
    text = open(os.path.join(REPO, "include", "smvp_cuda.h")).read()
    body = re.search(r"typedef struct %s\s*\{(.*?)\}\s*%s;" % (struct, struct), text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in filter(None, (d.strip() for d in body.split(";"))):
        _, declarators = decl.split(None, 1)  # every field type is one token (int32_t, int64_t)
        names += [re.match(r"\s*(\w+)", d).group(1) for d in declarators.split(",")]
    return names


def test_info_structs_match_the_header(tmp_path):
    """engine.py's ctypes mirrors of smvp_csr_info_t and smvp_tjds_info_t have the header's fields, offsets and size, as
    gcc lays the header out (no library build, no GPU)."""
    from smvp_toolkit_b200 import engine

    mirrors = {"smvp_csr_info_t": engine._CsrInfo, "smvp_tjds_info_t": engine._TjdsInfo}
    fields = {s: _header_fields(s) for s in mirrors}
    for s, py in mirrors.items():
        assert fields[s] == [f[0] for f in py._fields_], s
    src = ["#include <stddef.h>", "#include <stdio.h>", '#include "smvp_cuda.h"', "int main(void)", "{"]
    for s in mirrors:
        src.append('    printf("%s sizeof %%zu\\n", sizeof(%s));' % (s, s))
        src += ['    printf("%s %s %%zu\\n", offsetof(%s, %s));' % (s, f, s, f) for f in fields[s]]
    src += ["    return 0;", "}"]
    (tmp_path / "layout.c").write_text("\n".join(src) + "\n")
    exe = str(tmp_path / "layout")
    subprocess.run(["gcc", "-std=c11", "-I" + os.path.join(REPO, "include"), "-o", exe, str(tmp_path / "layout.c")], check=True)
    c = {tuple(ln.split()[:2]): int(ln.split()[2]) for ln in subprocess.run([exe], capture_output=True, text=True,
                                                                            check=True).stdout.splitlines()}
    for s, py in mirrors.items():
        assert c[(s, "sizeof")] == ctypes.sizeof(py), s
        for f in fields[s]:
            assert c[(s, f)] == getattr(py, f).offset, (s, f)


def test_time_stats_is_host_side(eng):
    td = eng.TimeData(np.array([1.0, 2.0, 3.0, 2.0]))
    assert td.time_total == 8.0 and td.time_avg == 2.0 and td.time_min == 1.0 and td.time_max == 3.0
    assert abs(td.time_stdev - np.sqrt(0.5)) < 1e-15


def test_product_never_touches_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py may use oracle/."""
    pkg = os.path.join(REPO, "smvp-toolkit_b200")
    for root, _, files in os.walk(pkg):
        if os.sep + "lib" in root:
            continue
        for f in files:
            if f.endswith((".py", ".c", ".h", ".cu", ".cuh")):
                text = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, re.M), f
                assert "libsmvp_oracle" not in text and "libsmvp_ref" not in text and "oracle/" not in text.replace(
                    "under oracle/", ""), f
    for so in ("libsmvp_cuda.so", "libsmvp_host.so"):
        p = os.path.join(pkg, "lib", so)
        if os.path.exists(p):
            out = subprocess.run(["ldd", p], capture_output=True, text=True).stdout
            assert "oracle" not in out and "smvp_ref" not in out
