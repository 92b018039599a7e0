"""GPU suite (-m gpu): the engine's option surface.  bpe_cuda_ctx_set_option accepts exactly the knobs listed
in include/bpe_cuda.h; the path-selecting switches the engine used to carry (in-place compaction, the streaming
kernel, forced census, speculative batches, programmatic dependent launch, L2 pinning) are gone, and their old
environment variables change nothing."""
import numpy as np
import pytest

from oracle_api import FAST_CF
from parity_cases import corpus

pytestmark = pytest.mark.gpu

# name -> the engine's default value
KNOBS = {"profile_replace": 0, "batch_steps": 64, "smem_hist_max_vocab": 448, "batch_max": 12, "batch_min_z": -1,
         "ranges": 0, "xchg_cap": 262144}
REMOVED = ["inplace", "use_stream", "force_census", "speculate", "pdl"]


@pytest.fixture
def ctx(engine):
    c = engine.Context(0)
    yield c
    c.close()


def test_remaining_knobs_are_accepted(ctx):
    for name, value in KNOBS.items():
        ctx.set_option(name, value)


@pytest.mark.parametrize("name", REMOVED)
def test_removed_knobs_are_unknown(ctx, name):
    with pytest.raises(ValueError):
        ctx.set_option(name, 0)


def test_removed_environment_variables_are_ignored(engine, oracle, monkeypatch):
    """1.5 MB is above the static limit, so the run takes the streaming kernel on the in-place RANGED layout."""
    for var, value in (("BPE_CUDA_INPLACE", "0"), ("BPE_CUDA_USE_STREAM", "0"), ("BPE_CUDA_PDL", "0"),
                       ("BPE_CUDA_SPECULATE", "0"), ("BPE_CUDA_L2_PIN", "1")):
        monkeypatch.setenv(var, value)
    data = corpus(0, 1_500_000, 5)
    rc, om, ot, _ = oracle.train(data, 200, FAST_CF)
    assert rc == 0 and len(om) == 200
    c = engine.Context(0)
    try:
        c.upload(data)
        c.train(200)
        m, t = c.download()
    finally:
        c.close()
    assert np.array_equal(m, om), "merge lists differ"
    assert np.array_equal(t, ot), "ids differ"
