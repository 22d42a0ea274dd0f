"""design_from_template on the device (micloc_design_templates, micloc_snn_design, micloc_hilbert_design,
micloc_design_vectors; SNNBeamformer / Beamformer.design_on_device).  Needs a B200: run with -m gpu.

Checked against the host design path on the same template: the delayed templates, the covariances, every solver mode
on crafted float64 matrices, the reference goldens, and the DoAs the designed matrices give on synthetic clips.

Tolerances (the largest errors measured on one B200 at its 1000 W power limit follow the table):
  templates against the host's float32 clips                        <= 1 float32 ulp
  covariance against the host path on the host's clips               DESIGN_REL 1e-8
  covariance against the same chain on the device's own clips        bit for bit
  mode 0 against _find_dc_removed_sing_vec (no sign alignment)       inf-norm 1e-6
  modes 1, 2 against numpy's SVD (top gap > 1e-3)                    |<u, u_host>| >= 1 - 1e-10
  mode 3 against scipy.linalg.eigh(a, b)                             |<u, u_host>| >= 1 - 1e-8
  designs against the host design on the same template               modes 1-3 |<>| >= 1 - 1e-8, mode 0 inf-norm 1e-6
Measured: templates 1 ulp at most (one value in 1.2e8 on the 64-mic linear array, all others bit-identical);
covariances against the host's 0; mode 0 7.5e-13; modes 1-3 and the designs 1 - |<>| below 1e-15; mode 0 designs 4.2e-13.
Mode 0's vector is orthogonal to the ones vector only as far as the bisection's rel_prec = 1e-8 converges (|1^T v| up
to 1.2e-3 measured, the host's of the same order): it is held to 10x the host's own value.
SNN bipolar: the chain's power depends on the phase of [Re u; Im u], and the phase rule (entry of largest modulus real)
picks a different phase than LAPACK; on 300 synthetic 10 dB clips 32 % of the DoA indices are identical to the host
matrix's, and the mean DoA error is 0.434 rad against the host's 0.485, so the test holds the device matrices to
localising as well as the host's (within 1.25x + one grid step).  On the c5_linear64 golden clip the device matrix gives
the neighbouring grid index.
Every matrix the solver takes is 2M x 2M (the real embedding of a complex M x M problem, or the SNN's 2M channels), so
the round-robin pair order always has an even size; odd n cannot reach it.
"""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.linalg import eigh

import helpers as H

pytestmark = pytest.mark.gpu

DESIGN_REL = 1e-8
MODE0_INF = 1e-6


def report(label, **errs):
    print(f"[design] {label}: " + ", ".join(f"{k}={v:.3e}" if isinstance(v, float) else f"{k}={v}"
                                            for k, v in errs.items()))


def lib():
    from haghighatshoarmuir2024_b200 import _native as N
    return N.lib()


def geometries():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray, LinearArray, Random2DArray
    np.random.seed(1)
    return {"center7": CenterCircularArray(4.5e-2, 7), "linear64": LinearArray(1e-2, 64, 0.32),
            "random64": Random2DArray(0.3, 64)}


def chirp(T, fs=48_000, f0=1600.0, f1=2400.0):
    t = np.arange(T) / fs
    return t, np.sin(2 * np.pi * (f0 + (f1 - f0) * t / t[-1] / 2) * t)


def snn_beamformer(geo, band, tau, bipolar, kernel_duration=10e-3, fs=48_000):
    from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
    b = SNNBeamformer(geo, kernel_duration, list(band), np.array([tau, tau]), bipolar_spikes=bipolar, fs=fs)
    b.verbose = False
    return b


def hilbert_beamformer(geo, band, fs=48_000):
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    b = Beamformer(geo, 10e-3, list(band), fs=fs)
    b.verbose = False
    return b


def resample(template, fs):
    t, s = template
    ti = np.arange(np.min(t), np.max(t), step=1 / fs)
    return ti, np.interp(ti, t, s)


def host_clips(beamf, ti, si, doa_list):
    return np.stack([beamf._delayed_template(ti, si, beamf.geometry.delays(theta=d, normalized=True))
                     for d in doa_list]).astype(np.float32)


def cplx(bf, M):
    return bf[:M] + 1j * bf[M:]


def phase_inner(a, b):
    """|<a_g, b_g>| per column of two unit-norm complex matrices [M, G]."""
    return np.abs(np.sum(np.conj(a) * b, axis=0))


def check_phase_rule(u):
    """Every complex column has a real positive entry of largest modulus.  (Entries whose moduli agree to 1e-12, such
    as the two coincident ring microphones of CenterCircularArray, are all candidates: rounding decides among them.)"""
    for g in range(u.shape[1]):
        a = np.abs(u[:, g])
        top = a >= a.max() * (1 - 1e-12)
        assert np.any(top & (u[:, g].imag == 0.0) & (u[:, g].real > 0.0)), g


# ---------------------------------------------------------------------------
# 1. templates
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name,T", [("center7", 4800), ("linear64", 2400), ("random64", 2400)])
def test_templates_match_the_host_interpolation(name, T):
    """micloc_design_templates against _delayed_template(...).astype(np.float32) and the Hilbert design loop's clips,
    on a grid of 512 DoAs from -pi to pi plus +-pi and 0 again: at most one float32 ulp apart."""
    geo = geometries()[name]
    beamf = snn_beamformer(geo, [1600, 2400], 2e-3, True)
    ti, si = resample(chirp(T), 48_000)
    doa_list = np.concatenate([np.linspace(-np.pi, np.pi, 512), [np.pi, -np.pi, 0.0]])
    eng = beamf.engine(np.zeros((2 * len(geo), 1)), ti)
    clips = eng.design_templates(geo, ti, si, doa_list).cpu().numpy()
    ref = host_clips(beamf, ti, si, doa_list)
    hil = []
    for doa in doa_list:                  # Beamformer.design_from_template's loop
        td = ti.reshape(-1, 1) - geo.delays(theta=doa, normalized=True).reshape(1, -1)
        td[td < ti.min()] = ti.min()
        hil.append(np.interp(td.ravel(), ti, si).reshape(td.shape))
    assert np.array_equal(ref, np.stack(hil).astype(np.float32))
    ulp = np.abs(clips.view(np.int32).astype(np.int64) - ref.view(np.int32).astype(np.int64))
    same = float(np.mean(ulp == 0))
    report(f"templates {name}", max_ulp=int(ulp.max()), bit_identical=same)
    assert ulp.max() <= 1


# ---------------------------------------------------------------------------
# 2. covariances
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("bipolar", [False, True])
def test_snn_design_covariance(bipolar):
    """cov_dev of micloc_snn_design: bit for bit SnnEngine.gram of the device's own clips / (T - T // 4), and within
    DESIGN_REL of the gram of the host's clips (what design_from_template computes)."""
    geo = geometries()["center7"]
    beamf = snn_beamformer(geo, [1600, 2400], 2e-3, bipolar)
    ti, si = resample(chirp(4800), 48_000)
    doa_list = np.linspace(-np.pi, np.pi, 64)
    T = len(ti)
    t0 = T // 4
    eng = beamf.engine(np.zeros((14, 1)), ti)
    bf, cov = eng.snn_design(geo, ti, si, doa_list, want_cov=True)
    n = torch.tensor(float(T - t0), dtype=torch.float64, device="cuda")      # a true division, as numpy's
    own = eng.gram(eng.design_templates(geo, ti, si, doa_list), t0) / n
    host = eng.gram(torch.from_numpy(host_clips(beamf, ti, si, doa_list)).cuda(), t0) / n
    torch.cuda.synchronize()
    assert torch.equal(cov, own)
    e = H.rel_err(cov.cpu().numpy(), host.cpu().numpy())
    report(f"snn cov bipolar={bipolar}", vs_host=e)
    assert e < DESIGN_REL


@pytest.mark.parametrize("M", [7, 16])
def test_hilbert_design_covariance(M):
    """cov_dev of micloc_hilbert_design: bit for bit SnnEngine.hilbert(bandpass=False) of the device's own clips, and
    within DESIGN_REL of design_from_template's covariance list (host clips)."""
    from haghighatshoarmuir2024_b200.array_geometry import CircularArray
    geo = CircularArray(4.5e-2, M)
    beamf = hilbert_beamformer(geo, [1600, 2400])
    t, s = chirp(4800)
    doa_list = np.linspace(-np.pi, np.pi, 48)
    ti, si = resample((t, s), 48_000)
    T, K = len(ti), len(beamf.kernel)
    t0 = min(K, T // 2)
    eng = beamf._engine()
    bf, cov = beamf.design_on_device((t, s), doa_list)
    raw = eng.hilbert(eng.design_templates(geo, ti, si, doa_list), t_start=t0, bandpass=False, want=("cov",))["cov"]
    own = torch.view_as_complex(torch.view_as_real(raw) * (1.0 / (T - t0)))      # numpy's complex / int
    _, host = beamf.design_from_template((t, s), doa_list)
    torch.cuda.synchronize()
    assert torch.equal(cov, own)
    e = H.rel_err(cov.cpu().numpy(), np.stack(host))
    report(f"hilbert cov M={M}", vs_host=e)
    assert e < DESIGN_REL


# ---------------------------------------------------------------------------
# 3. the solver alone
# ---------------------------------------------------------------------------
def psd(n, rng, rank=None, complex_=False):
    r = n if rank is None else rank
    X = rng.standard_normal((n, r + 3 if rank is None else r))
    if complex_:
        X = X + 1j * rng.standard_normal(X.shape)
    return X @ np.conj(X.T)


def with_spectrum(n, rng, lam, complex_=False):
    X = rng.standard_normal((n, n)) + (1j * rng.standard_normal((n, n)) if complex_ else 0)
    Q, _ = np.linalg.qr(X)
    return (Q * lam) @ np.conj(Q.T)


def crafted(n, rng, complex_=False):
    """random PSD, rank-deficient, a repeated bottom eigenvalue, closely spaced top eigenvalues"""
    out = [psd(n, rng, complex_=complex_), psd(n, rng, rank=max(2, n // 3), complex_=complex_)]
    lam = np.sort(rng.uniform(1, 2, n))[::-1]
    lam[n // 2:] = 0.5
    out.append(with_spectrum(n, rng, lam, complex_))
    lam = np.sort(rng.uniform(0, 1, n))[::-1]
    if n > 1:
        lam[0], lam[1] = 3.0, 3.0 - 1e-3
    out.append(with_spectrum(n, rng, lam, complex_))
    return np.stack([(A + np.conj(A.T)) / 2 for A in out])


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.parametrize("M", [1, 7, 32, 64])
def test_solver_mode0_is_the_dc_removed_vector(M):
    from haghighatshoarmuir2024_b200.engine import design_vectors
    from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
    rng = np.random.default_rng(M)
    Cs = crafted(2 * M, rng)
    got, root = design_vectors(0, dev(Cs), want_value=True)
    got = got.cpu().numpy()
    worst = worst_o = 0.0
    for g, Cm in enumerate(Cs):
        want = SNNBeamformer._find_dc_removed_sing_vec(None, Cm, rel_prec=1e-8)
        e = float(np.abs(got[:, g] - want).max())
        o = abs(float(np.sum(got[:, g])))
        worst, worst_o = max(worst, e), max(worst_o, o)
        assert e <= MODE0_INF, (g, e)
        assert o <= 10 * abs(float(np.sum(want))) + 1e-12, (g, o)
    report(f"mode 0 n={2 * M}", inf=worst, ones=worst_o)


@pytest.mark.parametrize("M", [1, 7, 32, 64])
def test_solver_mode1_is_the_top_singular_vector(M):
    from haghighatshoarmuir2024_b200.engine import design_vectors
    rng = np.random.default_rng(10 + M)
    Cs = crafted(2 * M, rng)
    got, sv = design_vectors(1, dev(Cs), want_value=True)
    u = cplx(got.cpu().numpy(), M)
    check_phase_rule(u)
    worst = 1.0
    for g, Cm in enumerate(Cs):
        A = (Cm[:M, :M] + Cm[M:, M:]) / 2 + 1j * (Cm[:M, M:] + Cm[M:, :M].T) / 2
        U, S, _ = np.linalg.svd(A)
        assert abs(float(sv[g]) - S[0]) <= 1e-10 * S[0]
        if M > 1 and (S[0] - S[1]) / S[0] <= 1e-3:
            continue
        d = float(np.abs(np.vdot(u[:, g], U[:, 0])))
        worst = min(worst, d)
        assert d >= 1 - 1e-10, (g, d)
    report(f"mode 1 M={M}", min_inner=worst)


@pytest.mark.parametrize("M", [1, 7, 64])
def test_solver_mode2_is_the_top_eigenvector(M):
    from haghighatshoarmuir2024_b200.engine import design_vectors
    rng = np.random.default_rng(20 + M)
    Cs = crafted(M, rng, complex_=True)
    got, lam = design_vectors(2, dev(Cs), want_value=True)
    u = got.cpu().numpy()
    check_phase_rule(u)
    worst = 1.0
    for g, Cm in enumerate(Cs):
        U, S, _ = np.linalg.svd(Cm)
        assert abs(float(lam[g]) - S[0]) <= 1e-10 * S[0]
        if M > 1 and (S[0] - S[1]) / S[0] <= 1e-3:
            continue
        d = float(np.abs(np.vdot(u[:, g], U[:, 0])))
        worst = min(worst, d)
        assert d >= 1 - 1e-10, (g, d)
    report(f"mode 2 M={M}", min_inner=worst)


@pytest.mark.parametrize("M,G", [(1, 4), (7, 8), (64, 6), (7, 1)])
def test_solver_mode3_is_the_generalised_eigenvector(M, G):
    """(G = 1 is interference removal with one DoA: C_sum - C_g is the diagonal loading alone.)"""
    from haghighatshoarmuir2024_b200.engine import design_vectors
    rng = np.random.default_rng(30 + M + G)
    Cs = np.stack([psd(M, rng, complex_=True) for _ in range(G)])
    got = design_vectors(3, dev(Cs)).cpu().numpy()
    check_phase_rule(got)
    Csum = sum(Cs)
    Csum = Csum + np.diag(np.mean(np.diag(Csum)) * np.ones(M)) / 10
    worst = 1.0
    for g, Cm in enumerate(Cs):
        w, V = eigh(Cm, Csum - Cm)
        v = V[:, -1] / np.linalg.norm(V[:, -1])
        if M > 1 and (w[-1] - w[-2]) / abs(w[-1]) <= 1e-3:
            continue
        d = float(np.abs(np.vdot(got[:, g], v)))
        worst = min(worst, d)
        assert d >= 1 - 1e-8, (g, d)
    report(f"mode 3 M={M} G={G}", min_inner=worst)


# ---------------------------------------------------------------------------
# 4. reference goldens, and the host design on the same template
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name,thr", [("snn_c1_bipolar", 0.999), ("snn_c5_linear64", 0.999),
                                      ("snn_c1_unipolar", 0.995), ("snn_c5_random64", 0.995)])
def test_snn_design_on_device_against_golden_and_host(name, thr):
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    g = H.load(name)
    M = len(g["r_vec"])
    fs = float(g["fs"])
    bipolar = bool(g["bipolar"])
    beamf = snn_beamformer(ArrayGeometry(g["r_vec"], g["theta_vec"]), g["band"], float(g["tau"]), bipolar,
                           kernel_duration=float(g["kernel_duration"]), fs=fs)
    t = np.arange(len(g["template"])) / fs
    bf = beamf.design_on_device((t, g["template"]), g["doa_list"])
    assert bf.is_cuda and bf.dtype == torch.float64 and bf.shape == g["bf_mat"].shape
    got = bf.cpu().numpy()
    host = beamf.design_from_template((t, g["template"]), g["doa_list"])
    if bipolar:
        u = cplx(got, M)
        check_phase_rule(u)
        gold = phase_inner(u, cplx(g["bf_mat"], M))
        vs_host = phase_inner(u, cplx(host, M))
        report(name, golden_min=float(gold.min()), host_min=float(vs_host.min()))
        assert gold.min() > thr
        assert vs_host.min() >= 1 - 1e-8
    else:
        gold = np.abs(np.sum(got * g["bf_mat"], axis=0))
        e = float(np.abs(got - host).max())
        report(name, golden_min=float(gold.min()), host_inf=e)
        assert gold.min() > thr
        assert e <= MODE0_INF
    x = torch.from_numpy(np.ascontiguousarray(g["x"], dtype=np.float32)).cuda().unsqueeze(0)
    doa = int(beamf.localize(got, np.arange(x.shape[1]) / fs, x)["doa"][0])
    G = got.shape[1]
    step = abs(doa - int(g["doa"]))
    if bipolar:                  # the bipolar chain's power depends on the columns' phase: a neighbouring index (c5)
        assert min(step, G - step) <= 1
    else:
        assert step == 0


@pytest.mark.parametrize("interference_removal", [False, True])
def test_hilbert_design_on_device_against_golden_and_host(interference_removal):
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    g = H.load("beamformer")
    beamf = hilbert_beamformer(CenterCircularArray(4.5e-2, 7), g["band"], fs=float(g["fs"]))
    t = np.arange(len(g["template"])) / float(g["fs"])
    bf, cov = beamf.design_on_device((t, g["template"]), g["doa_list"], interference_removal=interference_removal)
    assert bf.is_cuda and bf.dtype == torch.complex128 and cov.is_cuda and cov.dtype == torch.complex128
    u = bf.cpu().numpy()
    check_phase_rule(u)
    host, covs = beamf.design_from_template((t, g["template"]), g["doa_list"],
                                            interference_removal=interference_removal)
    vs_host = phase_inner(u, host)
    report(f"beamformer interference_removal={interference_removal}", host_min=float(vs_host.min()))
    assert vs_host.min() >= 1 - 1e-8
    xd = torch.from_numpy(g["x"]).cuda().unsqueeze(0)
    doa = int(beamf.localize(u, xd)["doa"][0])
    if interference_removal:                          # the golden holds the plain design
        assert doa == int(beamf.localize(host, xd)["doa"][0])
    else:
        assert phase_inner(u, g["bf_mat"]).min() >= 1 - 1e-6
        assert doa == int(g["doa"])


# ---------------------------------------------------------------------------
# 5. DoAs from device- and host-designed matrices on synthetic clips
# ---------------------------------------------------------------------------
def synthetic(geo, B, T, seed):
    from haghighatshoarmuir2024_b200.montecarlo import synthesize_clips
    rng = np.random.default_rng(seed)
    doa = rng.uniform(-np.pi, np.pi, B)
    return synthesize_clips(geo.r_vec, geo.theta_vec, 48_000, T, doa, snr_lin=np.full(B, 10.0), sine_freq=2000.0,
                            seed=seed), doa


def test_hilbert_matrices_localise_alike():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    geo = CenterCircularArray(4.5e-2, 7)
    beamf = hilbert_beamformer(geo, [1600, 2400])
    t, s = chirp(4800)
    doa_list = np.linspace(-np.pi, np.pi, 120, endpoint=False)
    dbf, _ = beamf.design_on_device((t, s), doa_list)
    hbf, _ = beamf.design_from_template((t, s), doa_list)
    x, _ = synthetic(geo, 300, 4800, 5)
    a = beamf.localize(dbf.cpu().numpy(), x)
    b = beamf.localize(hbf, x)
    pa, pb = a["power"].cpu().numpy(), b["power"].cpu().numpy()
    e = H.rel_err(pa, pb)
    report("hilbert synthetic power", rel=e)
    assert e < 1e-6
    da, db = a["doa"].cpu().numpy(), b["doa"].cpu().numpy()
    for i in np.nonzero(da != db)[0]:
        assert pb[i, da[i]] >= pb[i].max() * (1 - 1e-6), i


@pytest.mark.parametrize("bipolar", [False, True])
def test_snn_matrices_localise_alike(bipolar):
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    geo = CenterCircularArray(4.5e-2, 7)
    beamf = snn_beamformer(geo, [1600, 2400], 2e-3, bipolar)
    t, s = chirp(4800)
    G = 120
    doa_list = np.linspace(-np.pi, np.pi, G, endpoint=False)
    dbf = beamf.design_on_device((t, s), doa_list).cpu().numpy()
    hbf = beamf.design_from_template((t, s), doa_list)
    T = 4800
    x, truth = synthetic(geo, 300, T, 6)
    tv = np.arange(T) / 48_000
    a = beamf.localize(dbf, tv, x)
    b = beamf.localize(hbf, tv, x)
    da, db = a["doa"].cpu().numpy(), b["doa"].cpu().numpy()
    same = float(np.mean(da == db))
    step = np.abs(da - db)
    step = np.minimum(step, G - step)
    err = lambda d: float(np.mean(np.arcsin(np.abs(np.sin(doa_list[d] - truth)))))
    report(f"snn synthetic bipolar={bipolar}", identical=same, max_step=int(step.max()),
           within_2=float(np.mean(step <= 2)), doa_err_device=err(da), doa_err_host=err(db))
    if bipolar:
        # the SNN bipolar chain is not invariant under the columns' phase (header): the device's phase rule and
        # LAPACK's give different power; the matrices must localise as well as the host's
        assert err(da) <= 1.25 * err(db) + 2 * np.pi / G
    else:
        pb = b["power"].cpu().numpy()
        for i in np.nonzero(da != db)[0]:
            assert pb[i, da[i]] >= pb[i].max() * (1 - 1e-5), i


# ---------------------------------------------------------------------------
# 6. edges and ABI
# ---------------------------------------------------------------------------
def test_many_chunks_equal_the_per_chunk_results():
    """G = 2000 DoAs of a 1 s template at 7 microphones spans several chunks of both design calls; every slice of
    the DoA list designed on its own gives the same SNN columns and covariances bit for bit.  The Hilbert Gram path
    plans its time segments for the size of a chunk, so its float64 sums are grouped differently: covariances within
    1e-12, columns equal to 1 - 1e-10."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    geo = CenterCircularArray(4.5e-2, 7)
    ti, si = resample(chirp(48_000), 48_000)
    doa = np.linspace(-np.pi, np.pi, 2000)
    snn = snn_beamformer(geo, [1600, 2400], 2e-3, True)
    eng = snn.engine(np.zeros((14, 1)), ti)
    bf, cov = eng.snn_design(geo, ti, si, doa, want_cov=True)
    hil = hilbert_beamformer(geo, [1600, 2400])._engine()
    hbf, hcov = hil.hilbert_design(geo, ti, si, doa)
    for a, b in ((0, 170), (170, 1111), (1111, 2000)):
        pbf, pcov = eng.snn_design(geo, ti, si, doa[a:b], want_cov=True)
        assert torch.equal(pbf, bf[:, a:b]) and torch.equal(pcov, cov[a:b])
        qbf, qcov = hil.hilbert_design(geo, ti, si, doa[a:b])
        assert H.rel_err(qcov.cpu().numpy(), hcov[a:b].cpu().numpy()) < 1e-12
        assert phase_inner(qbf.cpu().numpy(), hbf[:, a:b].cpu().numpy()).min() >= 1 - 1e-10


def test_error_codes_and_launch_counts():
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray, CircularArray
    from haghighatshoarmuir2024_b200.engine import _design_template, design_vectors
    L = lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cov = torch.zeros((2, 14, 14), dtype=torch.float64, device="cuda")
    out = torch.zeros((14, 2), dtype=torch.float64, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    assert L.micloc_design_vectors(0, p(cov), 65, 2, p(out), None, 0, st) == N.ERR_UNSUPPORTED
    assert L.micloc_design_vectors(0, p(cov), 7, 0, p(out), None, 0, st) == N.ERR_SHAPE
    assert L.micloc_design_vectors(0, None, 7, 2, p(out), None, 0, st) == N.ERR_SHAPE
    assert L.micloc_design_vectors(0, p(cov), 7, 2, None, None, 0, st) == N.ERR_SHAPE
    assert L.micloc_design_vectors(4, p(cov), 7, 2, p(out), None, 0, st) == N.ERR_CONFIG
    assert L.micloc_design_vectors(-1, p(cov), 7, 2, p(out), None, 0, st) == N.ERR_CONFIG
    dev = torch.device("cuda", 0)
    doa = torch.zeros(3, dtype=torch.float64, device=dev)
    clips = torch.zeros((3, 100, 65), dtype=torch.float32, device=dev)
    tp, keep = _design_template(CircularArray(0.1, 65), np.arange(100) / 48e3, np.zeros(100), dev)
    assert L.micloc_design_templates(C.byref(tp), p(doa), 3, p(clips), 0, st) == N.ERR_UNSUPPORTED
    geo = CenterCircularArray(4.5e-2, 7)
    tp, keep = _design_template(geo, np.arange(1) / 48e3, np.zeros(1), dev)
    assert L.micloc_design_templates(C.byref(tp), p(doa), 3, p(clips), 0, st) == N.ERR_SHAPE
    tp, keep = _design_template(geo, np.arange(100) / 48e3, np.zeros(100), dev)
    assert L.micloc_design_templates(C.byref(tp), p(doa), 0, p(clips), 0, st) == N.ERR_SHAPE
    assert L.micloc_design_templates(C.byref(tp), None, 3, p(clips), 0, st) == N.ERR_SHAPE
    assert L.micloc_design_templates(C.byref(tp), p(doa), 3, None, 0, st) == N.ERR_SHAPE
    hil = hilbert_beamformer(geo, [1600, 2400])._engine()
    with pytest.raises(ValueError):                   # template of 6 microphones on a 7-microphone context
        hil.hilbert_design(CircularArray(0.1, 6), np.arange(100) / 48e3, np.zeros(100), [0.0])
    with pytest.raises(ValueError):
        hil.hilbert_design(geo, np.arange(100) / 48e3, np.zeros(99), [0.0])
    # launches: solver 1 (modes 0-2) / 3 (mode 3); Hilbert design of one chunk at M = 7: template + 3 (the analytic
    # signal's Gram path) + scale + solver
    spd = torch.from_numpy(crafted(14, np.random.default_rng(0))).cuda()
    for mode, n in ((0, 1), (1, 1)):
        l0 = L.micloc_launch_count()
        design_vectors(mode, spd)
        assert L.micloc_launch_count() - l0 == n
    hc = torch.from_numpy(crafted(7, np.random.default_rng(1), complex_=True)).cuda()
    for mode, n in ((2, 1), (3, 3)):
        l0 = L.micloc_launch_count()
        design_vectors(mode, hc)
        assert L.micloc_launch_count() - l0 == n
    ti, si = resample(chirp(4800), 48_000)
    for ir, n in ((False, 6), (True, 8)):
        l0 = L.micloc_launch_count()
        hil.hilbert_design(geo, ti, si, np.linspace(0, 1, 64), interference_removal=ir)
        assert L.micloc_launch_count() - l0 == n
    torch.cuda.synchronize()


def test_design_calls_do_not_synchronise():
    """With a long kernel queued ahead on the stream, micloc_hilbert_design and micloc_design_vectors return before
    it ends (inputs already on the device): nothing in them waits for the device.  The outputs are device tensors."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.engine import design_vectors
    geo = CenterCircularArray(4.5e-2, 7)
    hil = hilbert_beamformer(geo, [1600, 2400])._engine()
    ti, si = resample(chirp(4800), 48_000)
    td, sd = torch.from_numpy(ti).cuda(), torch.from_numpy(si).cuda()
    doa = torch.linspace(-np.pi, np.pi, 64, dtype=torch.float64, device="cuda")
    hil.hilbert_design(geo, td, sd, doa, interference_removal=True)        # warm: scratch allocated
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    for ir in (False, True):
        torch.cuda._sleep(int(2e9))
        bf, cov = hil.hilbert_design(geo, td, sd, doa, interference_removal=ir)
        assert not stream.query()
        v = design_vectors(3 if ir else 2, cov)
        assert not stream.query()
        assert bf.is_cuda and cov.is_cuda and v.is_cuda
        torch.cuda.synchronize()
        assert phase_inner(v.cpu().numpy(), bf.cpu().numpy()).min() >= 1 - 1e-12
