"""GPU: every output of the DDC bank, the PFB channelizer and the rational resampler, channel by channel, within its own
error bound (tests/bank_bounds.py, where the bounds are derived from each kernel's arithmetic) of an fp64 reference, on
every row of their tables: two calls on one handle through the device entry points, both kernel shapes, the library's
Kaiser prototypes, carriers 60 dB apart and batch rows 2^-20..2^20.  Row padding and the buffer around the rows stay
untouched, and the profiler (in a child process) sees the predicted instantiation for every call of the DDC rows (those of
the resampler and channelizer rows in their own files).

Each row prints `HEADROOM <row> <largest err / bound>`: how close the kernel comes to its bound."""
import os

import numpy as np
import pytest

import bank_bounds as bb
import kernel_variants as kv

pytestmark = pytest.mark.gpu

CASES = [(block, row) for block in ("resamp", "ddc", "pfb") for row in bb.block_rows(block)]


@pytest.mark.parametrize("block,row", CASES, ids=[bb.row_id(b, r) for b, r in CASES])
def test_every_output_within_its_bound(gpu, block, row):
    h, xs, ref, _ = bb.row_case(block, row)
    want = ref(h, xs)
    got = bb.run_row(gpu, block, row, h, xs, [w[0].shape[1] for w in want])
    worst = 0.0
    for k, ((y, clean), (yr, br, bi)) in enumerate(zip(got, want)):
        assert clean, (k, "wrote outside its output rows")
        assert y.shape == yr.shape, (k, y.shape, yr.shape)
        g = y.astype(np.complex128)
        er, ei = np.abs(g.real - yr.real) / br, np.abs(g.imag - yr.imag) / bi
        bad = (er > 1.0) | (ei > 1.0)
        if bad.any():
            c, m = np.argwhere(bad)[0]
            pytest.fail(f"call {k}: {int(bad.sum())} outputs beyond their bound, first channel {c} output {m}: got {g[c, m]}, "
                        f"want {yr[c, m]}, err / bound {er[c, m]:.3g} / {ei[c, m]:.3g}")
        worst = max(worst, float(er.max()), float(ei.max()))
    print(f"HEADROOM {bb.row_id(block, row)} {worst:.3g}")


def test_ddc_rows_launch_the_predicted_kernels(gpu):
    """The resampler's and the channelizer's rows are profiled in tests/test_gpu_resamp.py and tests/test_gpu_pfb.py."""
    got = kv.launched_in_child("ddc", int(os.environ.get("LOCAL_RANK", "0")))
    assert got == kv.predicted_launches("ddc")
