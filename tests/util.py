"""Helpers shared by the tests (test infrastructure; may use oracle/)."""
import os
import re

import numpy as np

from oracle import oracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
SAMPLES = ["ibm32", "curtis54", "pdp08-pg4", "memplus", "pwt"]

# golden report files shipped by the reference (SURVEY.md section 8c)
GOLDEN_REPORTS = {
    ("ibm32", "CSR"): "smvp-toolbox_report_CSR_1615284655.txt",
    ("memplus", "CSR"): "smvp-toolbox_report_CSR_1615284663.txt",
    ("pwt", "CSR"): "smvp-toolbox_report_CSR_1615284671.txt",
    ("curtis54", "CSR"): "smvp-toolbox_report_CSR_1615284695.txt",
    ("pdp08-pg4", "CSR"): "smvp-toolbox_report_CSR_1619162887.txt",
    ("ibm32", "TJDS"): "smvp-toolbox_report_TJDS_1615284655.txt",
    ("memplus", "TJDS"): "smvp-toolbox_report_TJDS_1615284665.txt",
    ("pwt", "TJDS"): "smvp-toolbox_report_TJDS_1615284679.txt",
    ("curtis54", "TJDS"): "smvp-toolbox_report_TJDS_1615284695.txt",
}


def sample_path(name):
    return os.path.join(GOLDEN, "sample-data", name + ".mtx")


def read_mtx_py(path):
    """Pure-python restatement of the reference's load loop (main-cli.c:1419-1441):
    1-based -> 0-based, pattern => val 1, symmetric files NOT expanded."""
    with open(path) as f:
        banner = f.readline().lower().split()
        pattern = banner[3] == "pattern"
        line = f.readline()
        while line.startswith("%"):
            line = f.readline()
        m, n, nnz = (int(t) for t in line.split())
        body = np.loadtxt(f, ndmin=2) if nnz else np.zeros((0, 3))
    coo = np.zeros(nnz, dtype=oracle.COO_DT)
    coo["row"] = body[:, 0].astype(np.int64) - 1
    coo["col"] = body[:, 1].astype(np.int64) - 1
    coo["val"] = 1.0 if pattern else body[:, 2]
    return m, n, coo


_cache = {}


def load_sample(name):
    if name not in _cache:
        _cache[name] = read_mtx_py(sample_path(name))
    return _cache[name]


def parse_report(path):
    """Parse a report in the reference's format (main-cli.c:294-316)."""
    with open(path) as f:
        lines = f.read().split("\n")
    out = {"header": lines[0]}
    for ln in lines:
        if ln.startswith("Non-zero numbers contained in matrix:"):
            out["nnz"] = int(ln.split(":")[1])
        if ln.startswith("Compute times for"):
            out["iters"] = int(ln.split()[3])
        for key, tag in (("total", "Total Time:"), ("avg", "Average Time:"), ("min", "Fastest Time:"),
                         ("max", "Slowest Time:"), ("stdev", "Time StDev:")):
            if ln.startswith(tag):
                out[key] = float(ln.split(":")[1].replace("ms", ""))
    a = lines.index("[")
    b = lines.index("]")
    out["y"] = np.array([float(t) for t in lines[a + 1:b]], dtype=np.float64)
    out["y_text"] = lines[a + 1:b]
    return out


def fmt_g(v):
    """C's %g for one double."""
    return "%g" % v


def rel_l2(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    d = np.linalg.norm(a - b)
    n = np.linalg.norm(b)
    return d / n if n > 0 else d


def random_coo(rng, m, n, nnz):
    cells = rng.choice(m * n, size=nnz, replace=False)
    coo = np.zeros(nnz, dtype=oracle.COO_DT)
    coo["row"] = cells // n
    coo["col"] = cells % n
    coo["val"] = rng.uniform(-1.0, 1.0, size=nnz)
    rng.shuffle(coo)
    return coo


# The store modes of the kernels that store y (YStore in csrc/common.cuh), as they appear in mangled kernel names
STORE_MODES = {"0": "Plain", "1": "Fanout", "2": "Axpby", "3": "Dot"}


def ystore(mode):
    """Regex fragment of a mangled template argument list that ends in store mode `mode` ("Plain", ... "Dot")."""
    return "LNS_6YStoreE%sEE" % {v: k for k, v in STORE_MODES.items()}[mode]


def store_modes(res_usage):
    """{kernel family: the set of store modes it is instantiated with}, from `cuobjdump -res-usage` output"""
    modes = {}
    for name, mode in re.findall(r"Function _ZN4smvp\d+(\w+?)I\w*?LNS_6YStoreE(\d)EEE", res_usage):
        modes.setdefault(name, set()).add(STORE_MODES[mode])
    return modes
