"""GPU test of the plan's lifetime: destroying a plan frees every device buffer it allocated.  The bounded
FFTFIT grid of pp_fit_phase_shift_batch_bounds (16 bytes per grid point) is one of them."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_plan_destroy_frees_the_bounded_grid_table():
    import torch
    from pulseportraiture_b200.engine import WidebandPlan

    rng = np.random.default_rng(11)
    profiles = rng.standard_normal((4, 64)).astype(np.float32)
    model = rng.standard_normal(64).astype(np.float32)
    ns = 1 << 20   # a 16 MB grid table per plan

    def cycle():
        with WidebandPlan(4, 64) as pl:
            r = pl.fit_phase_shift_batch(profiles, model, Ns=ns, bounds=(-0.25, 0.25))
        assert np.all(np.isfinite(r["phase"]))

    cycle()   # the first plan loads the kernels it launches, which takes device memory once
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for _ in range(8):
        cycle()
    torch.cuda.synchronize()
    free1 = torch.cuda.mem_get_info()[0]
    assert free0 - free1 < 32 << 20, "device free memory fell by %d bytes over 8 plans" % (free0 - free1)
