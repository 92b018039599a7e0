"""A sparse pass is two launches: the scan, then the delta application that also rewrites the stream.

Without a GPU: the statistics struct of include/bpe_cuda.h and its ctypes mirror agree field by field.  On the GPU: the
launch count of runs with sparse passes, a run whose speculative batches fall through, and encode on the sparse layout
reproducing the training ids."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import parity_cases as pc
from parity_cases import sha

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_stats_fields():
    src = open(os.path.join(ROOT, "include", "bpe_cuda.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    body = re.search(r"typedef struct\s*\{([^{}]*)\}\s*bpe_cuda_stats_t;", src).group(1)
    fields = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ctype, names = decl.split(None, 1)
        for n in names.split(","):
            n = n.strip()
            m = re.fullmatch(r"(\w+)\[(\d+)\]", n)
            fields.append((m.group(1), ctype, int(m.group(2))) if m else (n, ctype, 1))
    return fields


def test_stats_struct_matches_the_header():
    from llmtokenizer_b200._lib import Stats
    hdr = _header_stats_fields()
    py = Stats._fields_
    assert [f[0] for f in hdr] == [f[0] for f in py]
    size = {"uint64_t": 8, "double": 8}
    for (name, ctype, count), (pname, ptype) in zip(hdr, py):
        assert C.sizeof(ptype) == size[ctype] * count, name
        if ctype == "double":
            assert ptype is C.c_double, name
    assert C.sizeof(Stats) == sum(size[c] * k for _, c, k in hdr)
    for name in ("sparse_scan_ms", "dense_pass_ms", "convert_ms", "sparse_entries", "sparse_replacements"):
        assert name in Stats().as_dict()


# ---------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


def _train(engine, oracle, key):
    data, cap = pc.train_input(key)
    exp = pc.expected_train(key, oracle)
    ctx = engine.Context(0)
    try:
        ctx.upload(data)
        st = ctx.train(cap)
        m, t = ctx.download()
    finally:
        ctx.close()
    from test_gpu_parity import check_result
    check_result(exp, m, t, st, 1, key)
    return data, m, t, st


@gpu
@pytest.mark.parametrize("key", ["zipfa12m_10000", "uniform14m_2600"])
def test_two_launches_per_sparse_pass(engine, oracle, key):
    """Every merge step enqueues its pass launches and one delta application (dense layout: one pass kernel; sparse
    layout: the scan), so kernel_launches - 2 * steps counts what runs outside the steps: conversions, candidate lists,
    select-only launches, whole-table selections.  A sparse step of three or four launches would add at least one per
    sparse pass to it."""
    _, _, _, st = _train(engine, oracle, key)
    assert st["sparse_passes"] > 0, st
    outside = st["kernel_launches"] - 2 * st["replace_launches"]
    assert 0 <= outside < st["sparse_passes"], st
    assert 0 < st["sparse_replacements"] <= st["sparse_entries"], st


@gpu
def test_speculative_steps_that_fall_through_keep_the_result(engine, oracle):
    """Ties above the static limit pause the run; the batch enqueued behind the paused one falls through (its
    launches exit early) and the run still equals the oracle's."""
    _, _, _, st = _train(engine, oracle, "ties4m_1000")
    assert st["sparse_passes"] > 0 and st["same_bucket_ties"] > 0, st
    assert st["replace_launches"] > st["replace_passes"], st  # some enqueued steps ran no pass


@gpu
def test_encode_with_sparse_passes_reproduces_training(engine, oracle):
    data, m, t, st = _train(engine, oracle, "zipfb8m_2200")
    assert st["sparse_passes"] > 0, st
    ids, est = engine.encode(data, m)
    assert est["sparse_passes"] > 0, est
    assert len(ids) == len(t) and sha(np.asarray(ids)) == sha(t)
