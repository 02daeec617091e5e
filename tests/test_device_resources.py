"""Ownership of device memory in libkrotov_cuda: every cudaMalloc allocation and every CUDA IPC mapping is held by one
of the owning types of csrc/device_buffer.cuh, and a closed handle gives back all it took.

The structural checks read the sources (no GPU needed).  The GPU tests count the library's live allocations and
mappings (`krotov_live_device_objects`) around one short optimisation per kernel family: create, set_cheby, two
iterations, close."""
import os
import re

import numpy as np
import pytest

import krotov_jl_b200 as K
import workloads as W
from krotov_jl_b200.engine import KrotovCuda
from util import run_product

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "krotov.jl_b200", "csrc")


def _code(path):
    """Source without comments and string literals (error messages may name the CUDA calls they report)."""
    src = open(path).read()
    src = re.sub(r"//[^\n]*|/\*.*?\*/", "", src, flags=re.S)
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', src)


def _function(src, name):
    """Body of the function `name` (from its signature to the matching closing brace)."""
    m = re.search(r"\b" + name + r"\([^)]*\)\s*\{", src)
    assert m, name
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(src[i], 0)
        i += 1
    return src[m.start():i]


def test_only_the_owner_header_allocates_frees_or_unmaps():
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h")))
    assert "device_buffer.cuh" in sources
    for f in sources:
        calls = set(re.findall(r"\b(cudaMalloc\w*|cudaFree\w*|cudaIpcOpenMemHandle|cudaIpcCloseMemHandle)\b",
                               _code(os.path.join(CSRC, f))))
        if f == "device_buffer.cuh":
            assert calls == {"cudaMalloc", "cudaFree", "cudaIpcOpenMemHandle", "cudaIpcCloseMemHandle"}
        else:
            assert not calls, (f, calls)


def test_destroy_functions_name_no_buffer():
    host = _code(os.path.join(CSRC, "krotov_cuda.cu"))
    dense = _code(os.path.join(CSRC, "dense_kernel.cu"))
    for body in (_function(host, "krotov_destroy"), _function(dense, "dense_destroy")):
        assert not re.search(r"->\s*(d_\w+|cheb|peer_\w+|Hf|PSI|X|sw_\w+|graph_exec)\b", body), body
        assert "cudaFree" not in body and "release" not in body
    # the members that DenseEngine / krotov_handle_s own on the device are owning types, not raw pointers
    engine = re.search(r"struct DenseEngine \{(.*?)\n\};", dense, flags=re.S).group(1)
    assert not re.search(r"\b(double2|double|int|unsigned|long long)\s*\*\s*\w+\s*=\s*nullptr", engine)


def _calls(src, name):
    """The argument text of every call of `name` (balanced parentheses, across lines)."""
    out = []
    for m in re.finditer(r"\b" + name + r"\(", src):
        depth, i = 1, m.end()
        while depth:
            depth += {"(": 1, ")": -1}.get(src[i], 0)
            i += 1
        out.append(src[m.end():i - 1])
    return out


def test_every_device_write_is_ordered_on_the_handle_stream():
    """The sweeps run on the handle's non-blocking stream, which nothing orders after work on the legacy stream: every
    copy or memset that writes device memory is queued on the handle's stream (copy_to_device, cudaMemcpyAsync,
    cudaMemsetAsync).  Blocking cudaMemcpy stays only for device-to-host reads."""
    sources = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh")))
    assert {"krotov_cuda.cu", "dense_kernel.cu"} <= set(sources)
    for f in sources:
        src = _code(os.path.join(CSRC, f))
        assert not _calls(src, "cudaMemset"), f
        for args in _calls(src, "cudaMemcpy") + _calls(src, "cudaMemcpy2D"):
            assert "cudaMemcpyDeviceToHost" in args, (f, args)
        for args in _calls(src, "cudaMemcpyAsync") + _calls(src, "cudaMemsetAsync") + _calls(src, "copy_to_device"):
            if "cudaStream_t" not in args:  # (not the definition of copy_to_device)
                assert re.search(r",\s*(\w+->)?stream\s*(,|$)", args), (f, args)
    copies = _calls(_code(os.path.join(CSRC, "device_buffer.cuh")), "cudaMemcpyAsync")
    assert copies == ["dst, src, bytes, cudaMemcpyHostToDevice, stream"]


# ---- on the GPU ----------------------------------------------------------------------------------------------------
def _live():
    return K._lib.lib().krotov_live_device_objects()


def _nonlinear_c4():
    w = W.c4_ensemble(n_samples=8, n_grid=201)
    w.amp_poly = [[0.0, 1.0, 2.0]] + [None] * (w.L - 1)
    return w


def _dense_graph():
    w = W.dummy_dense(d=48, n_traj=12, n_controls=2, n_grid=41, seed=12)
    w.specrange = (-4.0, 4.0)  # fixed Chebyshev tables: the third identical iteration is captured, the fourth replayed
    return w


def _envelope_cb(wrk, it, *a):
    if it == 0:
        wrk.engine.envelope_extremes(np.array([[0.3, -0.2], [0.0, 0.0]]))


# (name, workload, iterations, run_product keywords, environment)
_FAMILIES = [
    ("tiny", W.c1_tls, 2, {}, {}),
    ("warp_c4", lambda: W.c4_ensemble(n_samples=8, n_grid=201), 2, {}, {}),
    ("pair", lambda: W.c4_ensemble(n_samples=12, n_grid=101), 2, {}, {"KROTOV_FORCE_PAIR": "1"}),
    ("seq_preg", lambda: W.c4_ensemble(n_samples=300, n_grid=41), 2, {}, {"KROTOV_SEQ_PREG": "1"}),
    ("wide64", lambda: W.c3_two_transmon(n_grid=41, levels=8, T=8.0), 2, {}, {}),
    ("wide128", lambda: W.c3_two_transmon(n_grid=41, levels=10, T=8.0), 2, {}, {}),
    ("ranks_replicate", lambda: W.c4_ensemble(n_samples=2, n_grid=101), 2,
     {"emulate_ranks": 2, "multi_gpu": "replicate"}, {}),
    ("ranks_shard", lambda: W.c4_ensemble(n_samples=2, n_grid=101), 2, {"emulate_ranks": 2, "multi_gpu": "shard"}, {}),
    ("dense_stream", lambda: W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=41, seed=11), 2, {"force_path": 2},
     {"KROTOV_NO_DSWEEP": "1"}),
    ("dense_cluster_sweep", lambda: W.dummy_dense(d=40, n_traj=6, n_controls=2, n_grid=41, seed=11), 2,
     {"force_path": 2}, {}),
    ("sparse_sweep", lambda: W.spin_chain(n_spins=6, n_traj=4, n_grid=21), 2, {"force_path": 3}, {}),
    ("dense_graph", _dense_graph, 4, {}, {"KROTOV_NO_DSWEEP": "1"}),
    ("nonlinear_amplitudes", _nonlinear_c4, 2, {}, {}),
    ("device_envelope", lambda: W.c4_ensemble(n_samples=24, n_grid=101), 2, {"callback": _envelope_cb}, {}),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,make,iters,kw,env", _FAMILIES, ids=[f[0] for f in _FAMILIES])
def test_close_gives_back_every_device_object(name, make, iters, kw, env, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    seen = {}

    def cb(wrk, it, *a):
        if "callback" in kw:
            kw["callback"](wrk, it, *a)
        seen["live"] = max(seen.get("live", 0), _live())

    base = _live()
    got = run_product(make(), iters, **{**kw, "callback": cb})
    assert seen["live"] > base  # the handle(s) did hold device memory while they were open
    assert _live() == base
    if name == "dense_graph":
        assert got["info"]["path"] == 2 and got["info"]["graph_replays"] >= 1
    if name.startswith("wide"):
        assert got["info"]["path"] == 1 and got["info"]["block_threads"] >= 64 + 32


@pytest.mark.gpu
def test_repeated_create_destroy_leaves_the_count_flat():
    w = W.c4_ensemble(n_samples=8, n_grid=201)
    counts = [_live()]
    for _ in range(3):
        run_product(w, 2)
        counts.append(_live())
    assert counts == [counts[0]] * 4


@pytest.mark.gpu
def test_refused_create_keeps_its_message_and_takes_nothing():
    w = W.c4_ensemble(n_samples=2, n_grid=21)
    base = _live()
    with pytest.raises(K.KrotovCudaError, match="lambda_a must be non-zero"):
        KrotovCuda(tlist=w.tlist, H0=w.H0, Hc=w.Hc, gen_of_traj=w.gen_of_traj, psi0=w.psi0, target=w.target,
                   update_shape=np.ones((w.L, len(w.tlist) - 1)), lambda_a=np.zeros(w.L), functional=K._lib.CHI_SM)
    assert b"lambda_a must be non-zero" in K._lib.lib().krotov_last_error(None)
    assert _live() == base
