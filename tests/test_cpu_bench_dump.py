"""bench.py --dump-outputs (no GPU): the arrays of a fit_batch call are written as <name>.npy in float32 /
float64, within 64 MB, every array keeping the same seeded sample of subints."""
import os

import numpy as np

import bench


def fake_results(nsub, nchan):
    """Arrays with fit_batch's names, shapes and dtypes; every element carries its subint index."""
    s = np.arange(nsub, dtype=np.float64)
    shapes = {"params": (5,), "param_errs": (5,), "nu_out": (3,), "cov": (5, 5), "chi2": (), "red_chi2": (),
              "snr": (), "phi_guess": (), "scales": (nchan,), "scale_errs": (nchan,), "channel_snrs": (nchan,),
              "noise": (nchan,)}
    res = {k: np.broadcast_to(s.reshape((nsub,) + (1,) * len(sh)), (nsub,) + sh).copy() for k, sh in shapes.items()}
    for k in ("nfeval", "return_code", "lag_index"):
        res[k] = np.arange(nsub, dtype=np.int32)
    res["noise"] = res["noise"].astype(np.float32)
    return res


def test_dump_samples_the_same_subints_within_budget(tmp_path):
    nsub = 10000                                  # the benchmark's batch: 147 MB of these arrays
    res = fake_results(nsub, 512)
    rows = bench.dump_outputs(res, nsub, str(tmp_path / "a"))
    assert 0 < rows < nsub
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(k + ".npy" for k in res)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    ref = None
    for k in res:
        got = np.load(tmp_path / "a" / (k + ".npy"))
        assert got.dtype == (np.float32 if k == "noise" else np.float64), k
        assert got.shape == (rows,) + res[k].shape[1:], k
        sub = got.reshape(rows, -1)[:, 0]
        assert np.all(got.reshape(rows, -1) == sub[:, None]), k
        ref = sub if ref is None else ref
        assert np.array_equal(sub, ref), k           # one sample of subints for every array
    assert np.all(np.diff(ref) > 0)
    bench.dump_outputs(res, nsub, str(tmp_path / "b"))
    for k in res:                                    # the sample is fixed: a second run writes the same rows
        assert np.array_equal(np.load(tmp_path / "a" / (k + ".npy")), np.load(tmp_path / "b" / (k + ".npy")))


def test_dump_writes_a_small_batch_whole(tmp_path):
    res = fake_results(64, 512)
    assert bench.dump_outputs(res, 64, str(tmp_path)) == 64
    for k, v in res.items():
        assert np.array_equal(np.load(tmp_path / (k + ".npy")), v), k
