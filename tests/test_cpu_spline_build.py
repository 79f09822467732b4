"""CPU checks of PCA / B-spline model building: the float64 numpy restatement of the device steps of
pplib.make_spline_model (used by tests/test_gpu_spline_build.py as the reference), the agreement of its Gram and
covariance routes, the write_spline_model -> read_spline_model round trip and the argument refusals."""
import numpy as np
import pytest

from oracle import pp_oracle as orc


# ---- restatement ------------------------------------------------------------------------------
def sign_convention(vecs):
    """columns with their entry of largest |value| (the first such) positive"""
    vecs = np.array(vecs, dtype=np.float64)
    ipk = np.argmax(np.abs(vecs), axis=0)
    return vecs * np.where(vecs[ipk, np.arange(vecs.shape[1])] < 0, -1.0, 1.0)


def moments(X, w, gram):
    """mu, and C = D^T D / W or G = D D^T / W with d_n = sqrt(w_n) (x_n - mu)"""
    W = w.sum()
    mu = (w[:, None] * X).sum(0) / W
    D = np.sqrt(w)[:, None] * (X - mu)
    return mu, (D @ D.T if gram else D.T @ D) / W


def moments_scale(X, w, gram):
    """sum_n w_n (|x_n| + |mu|)(|x_n| + |mu|)^T / W on the chosen side: the natural size of each entry's sum"""
    mu = (w[:, None] * X).sum(0) / w.sum()
    A = np.sqrt(w)[:, None] * (np.abs(X) + np.abs(mu))
    return (A @ A.T if gram else A.T @ A) / w.sum()


def basis(X, w, m, gram):
    """the top m unit eigenvectors [nbin, m] of the covariance, by either route, eigenvalues descending"""
    mu, M = moments(X, w, gram)
    vals, U = np.linalg.eigh(M)
    U = U[:, ::-1][:, :m]
    if gram:
        D = np.sqrt(w)[:, None] * (X - mu)
        U = D.T @ U
        U /= np.linalg.norm(U, axis=0)
    return vals[::-1][:m], sign_convention(U)


def find_kc(pows):
    """find_kc (pplib.py:1465-1495): scipy.optimize.brute's 20 x 20 x 20 np.mgrid (a slowest) of
    chi2 = sum_k (log10 pows_k - b e^{-a k} - dc)^2, np.argmin's choice (a NaN wins), then the first k with
    e^{-a k} < 0.005 (else nh - 1)"""
    y = np.log10(pows)
    nh = len(y)
    lo, hi = y.min(), y.max()
    grid = np.mgrid[nh ** -1.0:1.0:20j, 0:hi - lo:20j, lo:hi:20j].reshape(3, -1)
    k = np.arange(nh)
    c2 = np.empty(grid.shape[1])
    for i0 in range(0, grid.shape[1], 400):
        a, b, dc = grid[:, i0:i0 + 400, None]
        c2[i0:i0 + 400] = ((y - (b * np.exp(-a * k) + dc)) ** 2).sum(-1)
    nan = np.isnan(c2)
    i = int(np.nonzero(nan)[0][0]) if nan.any() else int(np.argmin(c2))
    hit = np.nonzero(np.exp(-grid[0, i] * k) < 0.005)[0]
    return int(hit[0]) if len(hit) else nh - 1


def lowpass(rows):
    """rfft, harmonics above find_kc's k_c zeroed (DC kept, Nyquist only when k_c = nbin/2), irfft"""
    rows = np.atleast_2d(rows)
    nbin = rows.shape[1]
    out, kcs = np.empty(rows.shape), np.empty(len(rows), dtype=int)
    for i, r in enumerate(rows):
        X = np.fft.rfft(r)
        kc = find_kc((X.real ** 2 + X.imag ** 2) / nbin)
        X[kc + 1:] = 0.0
        out[i], kcs[i] = np.fft.irfft(X, nbin), kc
    return out, kcs


def smooth_portrait(nchan, nbin, ncomp, seed, noise=0.01, zero=()):
    """a portrait of a Gaussian mean profile plus ncomp band-limited evolving components of decreasing size and
    white noise; channels in ``zero`` get weight 0"""
    rng = np.random.RandomState(seed)
    x = orc.get_bin_centers(nbin)
    f = np.linspace(-1, 1, nchan)
    port = np.exp(-0.5 * ((x - 0.4) / 0.03) ** 2)[None].repeat(nchan, 0)
    for j in range(ncomp):
        shape = np.exp(-0.5 * ((x - 0.4 - 0.02 * (j - 1)) / (0.02 + 0.01 * j)) ** 2) * np.cos(2 * np.pi * (j + 1) * x)
        port = port + (0.5 / (j + 1)) * np.sin(2.0 * f + j)[:, None] * shape[None]
    port = port + noise * rng.standard_normal(port.shape)
    w = rng.uniform(0.5, 2.0, nchan)
    w[list(zero)] = 0.0
    return port, w


# ---- tests ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("nchan,nbin", [(48, 64), (40, 100), (80, 64)])
def test_gram_and_covariance_routes_give_one_basis(nchan, nbin):
    port, w = smooth_portrait(nchan, nbin, 3, 7 * nchan + nbin, zero=(1, 5))
    vc, Ec = basis(port, w, 3, gram=False)
    vg, Eg = basis(port, w, 3, gram=True)
    assert np.allclose(vc, vg, rtol=1e-10, atol=0)
    assert np.all(np.sum(Ec * Eg, axis=0) >= 1 - 1e-12)


def test_lowpass_restatement_keeps_band_limited_rows():
    """a row whose power falls off smoothly to a floor keeps everything below k_c; k_c lands inside the band"""
    nbin = 512
    x = orc.get_bin_centers(nbin)
    r = np.exp(-0.5 * ((x - 0.5) / 0.02) ** 2) + 1e-6 * np.random.RandomState(3).standard_normal(nbin)
    out, kc = lowpass(r)
    assert 5 < kc[0] < nbin // 2
    X = np.fft.rfft(r)
    X[kc[0] + 1:] = 0
    assert np.array_equal(out[0], np.fft.irfft(X, nbin))
    assert np.abs(out[0] - r).max() < 1e-3


def test_write_spline_model_round_trip(tmp_path):
    import scipy.interpolate as si
    from pulseportraiture_b200 import pplib
    nbin = 256
    x = orc.get_bin_centers(nbin)
    mean_prof = np.exp(-0.5 * ((x - 0.3) / 0.02) ** 2)
    eigvec = np.linalg.qr(np.random.RandomState(2).standard_normal((nbin, 2)))[0]
    f = np.linspace(1200., 1800., 20)
    tck, _ = si.splprep(np.vstack([np.sin(f / 200.), np.cos(f / 300.)]), u=f, k=3, s=0)
    path = str(tmp_path / "m.spl")
    pplib.write_spline_model(path, "mdl", "J0000+0000", "data.npz", mean_prof, eigvec, tck, quiet=True)
    assert pplib.is_spline_model(path)
    name, src, df, mp, ev, tk = pplib.read_spline_model(path, quiet=True)
    assert (name, src, df) == ("mdl", "J0000+0000", "data.npz")
    assert np.array_equal(mp, mean_prof) and np.array_equal(ev, eigvec)
    assert np.array_equal(tk[0], tck[0]) and tk[2] == tck[2]
    freqs = np.linspace(1250., 1750., 8)
    _, model = pplib.read_spline_model(path, freqs, quiet=True)
    ref = np.dot(np.array(si.splev(freqs, tck)).T, eigvec.T) + mean_prof
    assert np.array_equal(model, ref)


def test_make_spline_model_refusals():
    from pulseportraiture_b200 import pplib
    port, w = smooth_portrait(8, 64, 1, 1)
    freqs = np.linspace(1200., 1800., 8)
    for k in (0, 6):
        with pytest.raises(ValueError, match="degree"):
            pplib.make_spline_model(port, freqs, k=k)
    dup = freqs.copy()
    dup[3] = dup[4]
    with pytest.raises(ValueError, match="duplicate"):
        pplib.make_spline_model(port, dup)
    wz = np.ones(8)
    wz[3] = 0.0
    few = np.zeros(8)
    few[:3] = 1.0
    with pytest.raises(ValueError, match="usable channels"):
        pplib.make_spline_model(port, freqs, weights=few, k=3)
    zero_rows = port.copy()
    zero_rows[3:] = 0.0
    with pytest.raises(ValueError, match="usable channels"):
        pplib.make_spline_model(zero_rows, freqs, k=3)
    with pytest.raises(ValueError, match="weights"):
        pplib.make_spline_model(port, freqs, weights=-wz)
    with pytest.raises(ValueError, match="freqs"):
        pplib.make_spline_model(port, freqs[:-1])
