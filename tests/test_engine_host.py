"""Host-side plumbing of the engine (GPU): a descriptor refused in a later chunk, and the wrap of the look-back epoch."""
import os

import numpy as np
import pytest

from gofr_b200 import _abi
from gofr_b200 import spec as S
from gofr_b200 import synth
from gofr_b200.table import Table
from tests import oracle as O
from tests.test_gpu_parity import DATE, _check

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "these tests need a GPU"
    return torch


def test_bad_descriptor_in_a_later_chunk(torch_cuda):
    """Request 3,500 of 5,000 points past the arena.  Every host-buffer call refuses its chunk (the fourth of 1,000) with
    GOFR_ERR_INVALID before launching it, while the chunks before it are in flight; the same engine then serves the intact
    batch exactly like the oracle."""
    from gofr_b200.engine import Engine, pin_batch, pinned_array
    spec = synth.config2_spec()
    batch = synth.config2_batch(5000)
    desc = batch.desc.copy()
    desc["arena_off"][3500] = batch.arena.size + 4096
    bad = S.RequestBatch(desc, batch.trace_ids, batch.arena)
    o1, f1, m1 = O.OracleTable(spec).serve(batch, DATE)
    n, total = batch.n, int(f1[-1])
    eng = Engine(Table(spec), 0)
    eng.set_chunk(1000)

    for pinned in (True, False):
        if pinned:   # device-driven egress
            good, wrong = pin_batch(batch), pin_batch(bad)
            out, off, meta = pinned_array(total + 64), pinned_array(4 * (n + 1), np.uint32), pinned_array(4 * n, np.uint32)
        else:        # pageable buffers: the exact-size copy pipeline
            good, wrong = batch, bad
            out, off, meta = np.zeros(total + 64, np.uint8), np.zeros(n + 1, np.uint32), np.zeros(n, np.uint32)
        with pytest.raises(_abi.GofrError) as err:
            eng.serve_host(wrong, DATE, out, off, meta)
        assert err.value.code == 1
        assert eng.serve_host(good, DATE, out, off, meta) == total
        assert np.array_equal(off, f1) and np.array_equal(meta, m1)
        assert out[:total].tobytes() == o1[:total].tobytes()

    slot = 544
    out, ln, meta = np.zeros(n * slot, np.uint8), np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    with pytest.raises(_abi.GofrError) as err:
        eng.serve_host_slots(bad, DATE, slot, out, ln, meta)
    assert err.value.code == 1
    eng.serve_host_slots(batch, DATE, slot, out, ln, meta)
    assert np.array_equal(ln, np.diff(f1.astype(np.int64)).astype(np.uint32)) and np.array_equal(meta, m1)
    assert (ln <= slot).all()
    rows, ob = out.reshape(n, slot), o1.tobytes()
    for i in range(n):
        assert rows[i, :ln[i]].tobytes() == ob[int(f1[i]):int(f1[i + 1])], i

    m2, v2 = O.route(O.OracleTable(spec), batch)
    with pytest.raises(_abi.GofrError) as err:
        eng.route_host(bad)
    assert err.value.code == 1
    m3, v3 = eng.route_host(batch)
    assert np.array_equal(m2, m3) and np.array_equal(v2, v3)
    eng.close()


def test_lookback_epoch_wrap(torch_cuda):
    """The engine starts its look-back epoch three launches before the 24-bit field wraps (GOFR_DEBUG_EPOCH_START is read
    once, when the engine is created).  Resident calls and chunked host calls, whose slots keep state words of their own,
    give the oracle's bytes on both sides of the wrap."""
    from gofr_b200.engine import Engine
    spec = synth.config2_spec()
    os.environ["GOFR_DEBUG_EPOCH_START"] = "0xFFFFFD"
    try:
        eng = Engine(Table(spec), 0)
    finally:
        del os.environ["GOFR_DEBUG_EPOCH_START"]
    # epochs 0xFFFFFE and 0xFFFFFF (two host chunks), the wrap to 1 (resident), 2..6 (five host chunks), 7, 8, 9..13
    for n, host in ((2000, True), (3000, False), (5000, True), (100, False), (9000, False), (5000, True)):
        _check(spec, synth.config2_batch(n, start=n), eng=eng, host=host, chunk=1000 if host else None)
    eng.close()
