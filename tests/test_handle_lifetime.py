"""Handles own every device allocation, pinned buffer, event and stream they create (common.cuh): a handle freed after
every lazily built member exists, and a build that fails after its staging buffers exist, leave this process's device
memory where it was.  The memory is NVML's per-process accounting, a read-only query: the GPU may be shared, so its
free memory says nothing about this process."""
import ctypes
import gc
import os
import warnings

import numpy as np
import pytest

import synth_ref
import util


def _process_device_bytes():
    """device memory NVML accounts to this process, summed over the devices; None when NVML does not list the process"""
    import pynvml

    pynvml.nvmlInit()
    try:
        total, seen = 0, False
        for i in range(pynvml.nvmlDeviceGetCount()):
            try:
                procs = pynvml.nvmlDeviceGetComputeRunningProcesses(pynvml.nvmlDeviceGetHandleByIndex(i))
            except pynvml.NVMLError:
                continue
            for p in procs:
                if p.pid == os.getpid():
                    seen = True
                    total += p.usedGpuMemory or 0
        return total if seen else None
    finally:
        pynvml.nvmlShutdown()


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def _with_wide_column(rng, m, nnz, long_col):
    """random m x m COO plus a column holding `long_col` entries: the transposed product then combines its partials"""
    coo = util.random_coo(rng, m, m, nnz)
    extra = np.zeros(long_col, dtype=coo.dtype)
    extra["row"] = np.arange(long_col)
    extra["col"] = 7
    extra["val"] = rng.uniform(-1, 1, long_col)
    keep = coo["col"] != 7
    return np.concatenate([coo[keep], extra])


def _csr_host_calls(eng, torch, monkeypatch, pattern):
    """a stencil large enough for the pipelined host call: pinned buffers, then pageable ones under SMVP_FORCE_OVERLAP,
    both equal to the device pass; the fused dot on both variants and the transposed handle"""
    lib = eng.lib()
    nx = 104
    m = nx ** 3
    r, c, v = eng.synth_stencil27(nx, nx, nx, value_mode=eng.VAL_STENCIL)
    A = eng.CsrMatrix.build_device(r, c, v, m, m, r.n)
    for a in (r, c, v):
        a.free()
    if not pattern:
        monkeypatch.setenv("SMVP_CSR_PATTERN", "0")
    dx = torch.empty(m, dtype=torch.float64, device="cuda")
    eng.synth_vector(dx, m, 5)
    dy = torch.empty(m, dtype=torch.float64, device="cuda")
    A.mult_device(dx, dy, eng.CSR_MERGE)
    torch.cuda.synchronize()
    monkeypatch.delenv("SMVP_CSR_PATTERN", raising=False)
    assert (A.row_patterns > 0) == pattern
    hx, hy = dx.cpu().pin_memory(), torch.zeros(m, dtype=torch.float64).pin_memory()
    ms = np.zeros(2)
    assert lib.smvp_csr_mult(A._h, ctypes.c_void_p(hx.data_ptr()), ctypes.c_void_p(hy.data_ptr()), 2,
                             ms.ctypes.data_as(ctypes.c_void_p), eng.CSR_MERGE) == eng.OK
    assert torch.equal(hy, dy.cpu())
    monkeypatch.setenv("SMVP_FORCE_OVERLAP", "1")
    y, _ = A.mult(dx.cpu().numpy(), iters=2, variant=eng.CSR_MERGE)
    monkeypatch.delenv("SMVP_FORCE_OVERLAP")
    assert np.array_equal(_bits(y), _bits(dy.cpu().numpy()))
    dd = torch.empty(1, dtype=torch.float64, device="cuda")
    for variant in (eng.CSR_MERGE, eng.CSR_VECTOR):
        A.mult_device_axpby_dot(2.0, dx, 0.5, dy, None, dd, variant)
    T = A.transpose()
    T.mult_device(dx, dy)
    torch.cuda.synchronize()
    T.free()
    A.free()


def _csr_small(eng, monkeypatch):
    """the pattern plan at fp32 and fp64, the batched `-n` loop, the tiny looping kernel and forced relabelling"""
    rng = np.random.default_rng(1)
    m = 12 ** 3
    for width in (4, 8):
        coo = synth_ref.stencil27(12, 12, 12)
        coo["val"] = rng.uniform(-1, 1, len(coo))
        if width == 4:
            coo["val"] = coo["val"].astype(np.float32).astype(np.float64)
        A = eng.CsrMatrix.build(coo, m, m)
        y1, _ = A.mult(np.ones(m), iters=1, variant=eng.CSR_MERGE)
        assert A.row_patterns == 27 and A.value_bytes == width
        y, _ = A.mult(np.ones(m), iters=50, variant=eng.CSR_MERGE)
        assert np.array_equal(_bits(y), _bits(y1))
        A.free()
    coo = synth_ref.stencil27(8, 8, 8)
    A = eng.CsrMatrix.build(coo, 512, 512)
    y1, _ = A.mult(np.ones(512), iters=1)
    y, _ = A.mult(np.ones(512), iters=20)
    assert np.array_equal(_bits(y), _bits(y1))
    A.free()
    monkeypatch.setenv("SMVP_CSR_RELABEL", "1")
    m = 40000
    x = rng.uniform(-1, 1, m)
    A = eng.CsrMatrix.build(util.random_coo(rng, m, m, 400000), m, m)
    y1, _ = A.mult(x, iters=1, variant=eng.CSR_MERGE)
    assert A.x_relabel == 1
    y, _ = A.mult(x, iters=8, variant=eng.CSR_MERGE)
    assert np.array_equal(_bits(y), _bits(y1))
    A.free()
    monkeypatch.delenv("SMVP_CSR_RELABEL")


def _tjds(eng, torch, monkeypatch, relabel):
    """every variant through the host call and the scaled / dot passes, then the transposed product of a handle with a
    column longer than TJDS_SEG^2 = 1024 entries, whose dot pass grows the dot scratch of the A x passes"""
    rng = np.random.default_rng(2)
    m = 30000
    monkeypatch.setenv("SMVP_TJDS_RELABEL", "1" if relabel else "0")
    A = eng.TjdsMatrix.build(_with_wide_column(rng, m, 300000, 3000), m, m)
    assert A.ndiag > 1024
    x = rng.uniform(-1, 1, m)
    dx = torch.as_tensor(x, device="cuda")
    dy = torch.zeros(m, dtype=torch.float64, device="cuda")
    dd = torch.empty(1, dtype=torch.float64, device="cuda")
    for variant in (eng.TJDS_ATOMIC, eng.TJDS_DETERMINISTIC, eng.TJDS_DETERMINISTIC_FAST):
        A.mult(x, iters=4, variant=variant)
        A.set_x_device(dx)
        A.mult_device_axpby(2.0, 0.5, dy, variant)
        A.mult_device_axpby_dot(2.0, 0.5, dy, None, dd, variant)
    assert A.y_relabel == (1 if relabel else -1)
    A.mult_transpose_device_axpby_dot(2.0, dx, 0.5, dy, None, dd)
    A.mult_transpose(x, iters=4)
    torch.cuda.synchronize()
    A.free()
    monkeypatch.delenv("SMVP_TJDS_RELABEL")


def _failed_builds(eng):
    """a coordinate out of range is found after the host COO has been staged on the device"""
    coo = synth_ref.stencil27(20, 20, 20)
    coo["row"][-1] = 8000
    for build in (eng.CsrMatrix.build, eng.TjdsMatrix.build):
        with pytest.raises(eng.SmvpError) as err:
            build(coo, 8000, 8000)
        assert err.value.code == eng.E_RANGE


def _round(eng, torch, monkeypatch):
    _csr_host_calls(eng, torch, monkeypatch, pattern=True)
    _csr_host_calls(eng, torch, monkeypatch, pattern=False)
    _csr_small(eng, monkeypatch)
    for relabel in (False, True):
        _tjds(eng, torch, monkeypatch, relabel)
    _failed_builds(eng)
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_freed_handles_return_their_device_memory(monkeypatch):
    import torch

    import smvp_toolkit_b200 as eng

    _round(eng, torch, monkeypatch)  # loads every module and warms the allocators
    start = _process_device_bytes()
    after = []
    for _ in range(3):
        _round(eng, torch, monkeypatch)
        after.append(_process_device_bytes())
    if start is None:
        warnings.warn("NVML does not list this process: the lifecycle ran without its memory check")
        return
    assert after == [start] * len(after), (start, after)
