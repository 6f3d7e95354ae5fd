"""Error convention of the C-ABI on a GPU box: infrastructure errors are negative MULLS_E_* codes with a message
from mulls_last_error, distinct from the algorithmic process code; nothing falls back silently."""
import numpy as np
import pytest

from mulls_b200 import abi

pytestmark = pytest.mark.gpu


def test_capacity_unsupported_and_state_errors(small_pair):
    from mulls_b200.registration import Context

    ctx = Context(0, 1, 1000, 1000)
    with pytest.raises(RuntimeError, match="-102"):       # MULLS_E_CAPACITY: pair larger than the context
        ctx.run_batch([small_pair])
    with pytest.raises(RuntimeError, match="-102"):       # more pairs than max_pairs
        ctx.run_batch([small_pair, small_pair])
    ctx.close()
    ctx = Context(0, 1, 100000, 100000)
    with pytest.raises(RuntimeError, match="-101"):       # MULLS_E_ARG: nothing uploaded
        ctx.run_resident()
    p = abi.IcpParams.from_buffer_copy(small_pair["params"])
    p.max_iter_num = 1000
    with pytest.raises(RuntimeError, match="-101"):
        ctx.run_batch([dict(small_pair, params=p)])
    res, _ = ctx.run_batch([small_pair])                  # the context is still usable after errors
    assert res[0]["code"] == 1
    ctx.close()


def test_threshold_schedule_out_of_range(small_pair):
    """the threshold schedule sizes the search grid: a non-finite or non-positive dis_thre_unit / dis_thre_update_rate,
    or a negative / non-finite dis_thre_min, is MULLS_E_ARG; h0_min_mm <= 0 too"""
    from mulls_b200.registration import Context

    ctx = Context(0, 1, 100000, 100000)
    bad = [("dis_thre_unit", v) for v in (0.0, -1.5, float("nan"), float("inf"))]
    bad += [("dis_thre_update_rate", v) for v in (0.0, -1.1, float("nan"), float("inf"))]
    bad += [("dis_thre_min", v) for v in (-0.1, float("nan"), float("inf"))]
    for name, v in bad:
        p = abi.IcpParams.from_buffer_copy(small_pair["params"])
        setattr(p, name, v)
        with pytest.raises(RuntimeError, match="-101"):
            ctx.run_batch([dict(small_pair, params=p)])
    with pytest.raises(RuntimeError, match="-101"):
        ctx.set_tunable("h0_min_mm", 0)
    p = abi.IcpParams.from_buffer_copy(small_pair["params"])
    p.dis_thre_min = 0.0                                  # the edges that stay valid
    res, _ = ctx.run_batch([dict(small_pair, params=p)])
    assert res[0]["code"] == 1
    ctx.close()
