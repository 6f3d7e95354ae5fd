"""mulls_set_tunable on a GPU box: the names it accepts and the values it rejects, on a single, a native pipelined and
a Python pipelined context; and the twin context a one-shot batch is double-buffered over, which must run with the
tunables of its context however they were set."""
import numpy as np
import pytest

from mulls_b200 import abi

pytestmark = pytest.mark.gpu

DEFAULTS = {"leaf_count": 32, "hash_slack": 4, "h0_min_mm": 125, "use_graph": 1, "loop_kernel": 1, "host_pack": 2,
            "pack_threads": 0}
RETIRED = {"start_level": 5, "defer_from_iter": 3, "reseed_cells_x4": 16, "search_blocks": 12, "sort_sources": 1,
           "zero_copy": 0, "stage_wc": 0, "poll_pause": 64, "double_buffer": 1, "pairs_in_flight": 1}
OUT_OF_RANGE = [("use_graph", 2), ("use_graph", -1), ("loop_kernel", 2), ("loop_kernel", -1), ("host_pack", 3),
                ("host_pack", -1)]


def handles(ctx):
    return [c.handle for c in ctx.lanes] if hasattr(ctx, "lanes") else [ctx.handle]


def test_names_and_values():
    from mulls_b200.registration import Context, PipelinedContext

    lib = abi.load_library()
    ctxs = [Context(0, 2, 20000, 20000), Context(0, 2, 20000, 20000, lanes=2), PipelinedContext(0, 2, 1, 20000, 20000)]
    try:
        for ctx in ctxs:
            for h in handles(ctx):
                for name, value in DEFAULTS.items():
                    assert lib.mulls_set_tunable(h, name.encode(), value) == 0, name
                for name, value in list(RETIRED.items()) + OUT_OF_RANGE:
                    assert lib.mulls_set_tunable(h, name.encode(), value) == abi.E_ARG, (name, value)
    finally:
        for ctx in ctxs:
            ctx.close()


def test_twin_takes_tunables_set_before_it_exists(small_pair):
    """A batch of four pairs runs as two halves, on the context and on its twin (created by the first such call).
    loop_kernel = 0 set before the twin exists must hold for the twin as it does when set after."""
    from mulls_b200.registration import Context

    pairs = [small_pair] * 4
    a = Context(0, 4, 100000, 100000)
    b = Context(0, 4, 100000, 100000)
    try:
        a.set_tunable("loop_kernel", 0)
        ra, _ = a.run_batch(pairs)
        sa = a.stats()
        b.run_batch(pairs)
        b.set_tunable("loop_kernel", 0)
        rb, _ = b.run_batch(pairs)
        sb = b.stats()
        assert sa["kernel_launches"] == sb["kernel_launches"]
        for x, y in zip(ra, rb):
            for k in x:
                np.testing.assert_array_equal(np.asarray(x[k]), np.asarray(y[k]), err_msg=k)
    finally:
        a.close()
        b.close()
