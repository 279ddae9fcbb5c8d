"""The slab path's unfit-row counts reach the host without a copy in the stream: the last CTA of the table and of the
hist kernel stores them into the pinned status mirror, and the hist kernel's last CTA resets the device counters for
the next call.  Calls that alternate between fit rows, a few unfit rows and tie-heavy rows in one context must each
take their own route and give the part pipeline's counts, so that no count leaks from one call into the next."""
import numpy as np
import pytest


def _crowded_row(rng, n):
    """Distinct values where the table kernel samples (64 chunks of 256 consecutive values, mbd_slab.cuh) and a crowd
    within 1e-9 of zero everywhere else: thousands of values in one bin, which the hist kernel's validation rejects."""
    x = 1e-9 * rng.random(n)
    gap = (n - 256) // 63
    for c in range(64):
        x[c * gap:c * gap + 256] = rng.standard_normal(256)
    return x


def _matrices(n, T):
    rng = np.random.default_rng(9100)
    fit = rng.standard_normal((T, n)).cumsum(0)
    few = rng.standard_normal((T, n))   # 2 of 40 rows: the hist kernel's validation gives them up
    few[4] = _crowded_row(rng, n)
    few[31] = _crowded_row(rng, n)
    ties = np.round(rng.standard_normal((T, n)), 2)  # every row: the table kernel's sample sees the ties
    return {"fit": fit, "few": few, "ties": ties}


@pytest.mark.gpu
def test_slab_counts_do_not_leak_between_calls(engine, monkeypatch):
    import torch
    n, T = 20_000, 40
    dev = torch.device("cuda", 0)
    mats = {k: torch.from_numpy(v).to(dev) for k, v in _matrices(n, T).items()}
    out = torch.zeros(n, dtype=torch.int64, device=dev)

    def counts(X):
        engine.band_depth_counts_dev(X.data_ptr(), T, n, n, out.data_ptr(), None, n, 2, True)
        return out.cpu().numpy().copy(), engine.timings()["launches"]

    monkeypatch.setenv("SD_MBD_PATH", "parts")
    want, parts_launches = {}, {}
    for k, X in mats.items():
        want[k], parts_launches[k] = counts(X)
    monkeypatch.delenv("SD_MBD_PATH")
    # device-resident calls wait for both counts: table + hist + rank + finish when every row fits; the rank kernel
    # and the masked part pipeline when a few rows do not; the whole part pipeline after the table and hist kernels
    # when many rows do not
    route_launches = {"fit": 4, "few": parts_launches["few"] + 3, "ties": parts_launches["ties"] + 2}
    for k in ("fit", "few", "fit", "ties", "fit", "ties", "few", "few", "fit"):
        got, launches = counts(mats[k])
        assert np.array_equal(got, want[k]), k
        assert launches == route_launches[k], (k, launches, route_launches[k])
