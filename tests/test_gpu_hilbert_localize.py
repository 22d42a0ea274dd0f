"""The Hilbert beamformer at batch scale (micloc_hilbert_localize, Beamformer.localize / design_from_template,
SnrSweep.run_band_hilbert).  Needs a B200: run with -m gpu.

Power, DoA and the design covariance come from the real Gram matrix G = sum_{t >= t_start} z_t z_t^T of the analytic
signal z = [Re s | Im s].  They are checked against a float64 restatement built from the call's own `z` tap:

  cov64    = (Grr + Gii) + i (Gri - Gir) = S^H S over rows t >= t_start
  power64  = mean_{t >= t_start} |s_t . conj(bf_g)|^2
  doa      = the first maximum of power64 (check_doa of test_gpu_power_paths: near-ties within the tolerance pass)

Tolerances, with the largest error measured on one B200 (1000 W power limit) in brackets.  The new bounds are about 10x
that error; the float64, float32-projection and front-end bounds are the existing ones of test_gpu_power_paths.py and
test_gpu_parity.py:
  M <= 8, k_hilbert_gram (float64 products and sums): cov, relative to the clip's largest |cov|   1e-12  (4.2e-14)
                                                        power, excess over float32 rounding          1e-12  (0)
  M > 8, k_gram_tiled (float32 over 1024-sample slabs, float64 across slabs): cov and power        5e-6   (5.2e-7)
  segmented clip (B = 1, T = 480 000): z against the sequential z of run_taps, of max |z|           4e-5   (3.6e-6)
  design covariance against the old per-DoA loop (float64 roll part there, float32 here)            1e-8   (9.0e-10)
  power against micloc_hilbert_beamform (float32 projections)                                      4e-6   (8.2e-8)
  power against the oracle's beamformer_apply (the front-end tolerance)                             1e-4   (3.0e-6)
The z tap on the sequential plan equals run_taps' z tap bit for bit (same kernels, same arithmetic).
"""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.signal import sosfilt

import helpers as H
import test_gpu_power_paths as PP

pytestmark = pytest.mark.gpu

GRAM64 = 1e-12
TILED_REL = 5e-6
SEG_Z_REL = 4e-5
DESIGN_REL = 1e-8
DENSE_REL = 4e-6


def steering(M, G, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((M, G)) + 1j * rng.standard_normal((M, G))


def restate(z, W, t_start):
    """(cov64 [B,M,M] complex, power64 [B,G]) of z [B,T,2M] over rows t >= t_start."""
    M = W.shape[0]
    v = np.asarray(z, np.float64)[:, t_start:]
    s = v[..., :M] + 1j * v[..., M:]
    cov = np.einsum("bti,btj->bij", np.conj(s), s)
    power = np.mean(np.abs(s @ np.conj(W)) ** 2, axis=1)
    return cov, power


def cov_err(cov, ref):
    return PP.rel_err(torch.view_as_real(cov).cpu().numpy(), np.stack([ref.real, ref.imag], -1))


def hilbert_engine(M, G, seed=0):
    g = PP.array_case(M, 4)
    eng = PP.engine(g, 4801)             # (the neuron constants of the spec are not used by the Hilbert path)
    W = steering(M, G, seed)
    eng.set_hilbert_bf(W)
    return g, eng, W


def check_against_own_z(eng, xd, W, t_starts, tol, label):
    """One call with the z tap, then every t_start without it: cov, power and DoA against the restatement."""
    z = eng.hilbert(xd, want=("z",))["z"].cpu().numpy()
    worst_c = worst_p = 0.0
    for t0 in t_starts:
        out = eng.hilbert(xd, t_start=t0, want=("cov", "power", "doa"))
        torch.cuda.synchronize()
        cov64, p64 = restate(z, W, t0)
        ec = cov_err(out["cov"], cov64)
        p = out["power"].cpu().numpy()
        ep = PP.f64_excess(p, p64) if tol == GRAM64 else PP.rel_err(p, p64)
        worst_c, worst_p = max(worst_c, ec), max(worst_p, ep)
        assert ec < tol, (t0, ec)
        assert ep < tol, (t0, ep)
        PP.check_doa(out["doa"].cpu().numpy(), p64, tol)
    PP.report(label, cov=worst_c, power=worst_p)
    return z


# ---------------------------------------------------------------------------
# 1. reference golden
# ---------------------------------------------------------------------------
def test_localize_and_design_match_reference_golden():
    """Beamformer.localize on the golden clip: the golden DoA and power within 1e-4; design_from_template on the
    golden template: every column equals the golden bf_mat up to phase, and localising with it gives the golden DoA."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    g = H.load("beamformer")
    bf = Beamformer(CenterCircularArray(4.5e-2, 7), 10e-3, list(g["band"]), fs=float(g["fs"]))
    bf.verbose = False
    xd = torch.from_numpy(g["x"]).cuda().unsqueeze(0)
    out = bf.localize(g["bf_mat"], xd)
    torch.cuda.synchronize()
    assert int(out["doa"][0]) == int(g["doa"])
    assert H.rel_err(out["power"][0].cpu().numpy(), g["power"]) < 1e-4
    T = len(g["template"])
    t = np.arange(T) / float(g["fs"])
    bf_mat, covs = bf.design_from_template((t, g["template"]), g["doa_list"])
    assert bf_mat.shape == g["bf_mat"].shape and len(covs) == len(g["doa_list"])
    inner = np.abs(np.sum(np.conj(bf_mat) * g["bf_mat"], axis=0))
    assert inner.min() >= 1 - 1e-6, inner.min()
    assert int(bf.localize(bf_mat, xd)["doa"][0]) == int(g["doa"])
    with pytest.raises(ValueError, match="number of channels"):
        bf.localize(g["bf_mat"], xd[..., :6])


# ---------------------------------------------------------------------------
# 2. exact arithmetic against the call's own z tap
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("int16", [False, True])
@pytest.mark.parametrize("M", [1, 2, 7, 8, 16, 64])
def test_cov_power_doa_equal_restatement_of_own_z(M, int16):
    """M <= 8 (k_hilbert_gram, float64) and M = 16, 64 (z + k_gram_tiled): T in {1, 100, 4801, 48000}, t_start in
    {0, 1, T // 4, T - 1}, B = 3 (B = 2 at T = 48000)."""
    G = 37
    for T in (1, 100, 4801, 48_000):
        B = 2 if T == 48_000 else 3
        g, eng, W = hilbert_engine(M, G, seed=M + T)
        x = PP.clips(g, B, T, seed=M + T, int16=int16)
        tol = GRAM64 if M <= 8 else TILED_REL
        check_against_own_z(eng, PP.to_dev(x), W, sorted({0, min(1, T - 1), T // 4, T - 1}), tol,
                            f"hilbert M={M} T={T} int16={int16}")
        eng.close()


@pytest.mark.parametrize("M", [7, 64])
def test_segmented_long_clip(M, monkeypatch):
    """B = 1, T = 480 000 (ten seconds) runs in time segments with a band-pass warm-up: cov / power / DoA exact against
    its own z; z within SEG_Z_REL of the sequential z of run_taps."""
    T, G = 480_000, 37
    g, eng, W = hilbert_engine(M, G, seed=3)
    xd = PP.to_dev(PP.clips(g, 1, T, seed=5))
    z = check_against_own_z(eng, xd, W, [0, T // 4], GRAM64 if M <= 8 else TILED_REL, f"segmented M={M}")
    monkeypatch.setenv("MICLOC_NO_SEGMENTS", "1")       # run_taps on the sequential plan
    zs = eng.run_taps(xd, want=("z",))["z"].cpu().numpy()
    err = PP.rel_err(z, zs)
    PP.report(f"segmented z M={M}", vs_sequential=err)
    assert 0 < err < SEG_Z_REL           # (> 0: the segmented plan did run)


def test_batch_beyond_65535_clips():
    """B = 70 000 short clips: chunks of at most 65 535, each clip's results at its own index."""
    M, T, G, B = 2, 64, 9, 70_000
    g, eng, W = hilbert_engine(M, G, seed=1)
    x = np.random.default_rng(2).standard_normal((B, T, M)).astype(np.float32)
    xd = PP.to_dev(x)
    out = eng.hilbert(xd, t_start=3, want=("z", "cov", "power", "doa"))
    torch.cuda.synchronize()
    cov64, p64 = restate(out["z"].cpu().numpy(), W, 3)
    assert cov_err(out["cov"], cov64) < GRAM64
    assert PP.f64_excess(out["power"].cpu().numpy(), p64) < GRAM64
    PP.check_doa(out["doa"].cpu().numpy(), p64, GRAM64)


# ---------------------------------------------------------------------------
# 3. front end
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("M", [7, 16])
def test_front_end_z_and_design_cov(M):
    """z tap = run_taps' z tap bit for bit, and within the STHT tolerance of scipy float64 (sosfilt of roll + STHT);
    bandpass=0: cov = S^H S of roll(x) + j q with q the STHT tap of run_taps."""
    T, B = 4801, 3
    g, eng, W = hilbert_engine(M, 5)
    x = PP.clips(g, B, T, seed=11)
    xd = PP.to_dev(x)
    z = eng.hilbert(xd, want=("z",))["z"].cpu().numpy()
    tap = eng.run_taps(xd, want=("q", "z"))
    assert np.array_equal(z, tap["z"].cpu().numpy())
    K = len(g["kernel"])
    x64 = x.astype(np.float64)
    q64 = np.stack([np.stack([np.convolve(x64[b, :, m], g["kernel"])[:T] for m in range(M)], -1) for b in range(B)])
    sos = eng.spec.sos
    z64 = sosfilt(sos, np.concatenate([np.roll(x64, K // 2, axis=1), q64], -1), axis=1)
    assert PP.rel_err(z, z64) < 1e-4
    t0 = min(K, T // 2)
    cov = eng.hilbert(xd, t_start=t0, bandpass=False, want=("cov",))["cov"]
    s = np.roll(x64, K // 2, axis=1) + 1j * tap["q"].cpu().numpy().astype(np.float64)
    s = s[:, t0:]
    ref = np.einsum("bti,btj->bij", np.conj(s), s)
    e = cov_err(cov, ref)
    PP.report(f"design cov M={M}", rel=e)
    assert e < (GRAM64 if M <= 8 else TILED_REL)


@pytest.mark.parametrize("interference_removal", [False, True])
def test_design_equals_per_doa_loop(interference_removal):
    """design_from_template against the per-DoA loop it replaces (run_taps' q tap, numpy covariance), with and without
    interference removal: covariances within DESIGN_REL, steering columns equal up to phase."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    fs, T, G = 48_000, 4800, 40
    bf = Beamformer(CenterCircularArray(4.5e-2, 7), 10e-3, [1600, 2000], fs=fs)
    bf.verbose = False
    t = np.arange(T) / fs
    src = np.sin(2 * np.pi * (1600 + 400 * t / t[-1]) * t)
    doa_list = np.linspace(-np.pi, np.pi, G)
    bf_mat, covs = bf.design_from_template((t, src), doa_list, interference_removal=interference_removal)
    eng = bf._engine()
    K = len(bf.kernel)
    ti = np.arange(t.min(), t.max(), 1 / fs)
    si = np.interp(ti, t, src)
    ref = []
    for doa in doa_list:
        td = ti.reshape(-1, 1) - bf.geometry.delays(theta=doa, normalized=True).reshape(1, -1)
        td[td < ti.min()] = ti.min()
        sv = np.interp(td.ravel(), ti, si).reshape(td.shape)
        q = eng.run_taps(torch.from_numpy(sv.astype(np.float32)).cuda(), want=("q",))["q"][0].cpu().numpy()
        sh = np.roll(sv, K // 2, axis=0) + 1j * q.astype(np.float64)
        st = sh[min(K, sh.shape[0] // 2):]
        ref.append(st.conj().T @ st / st.shape[0])
    err = max(float(np.abs(c - r).max() / np.abs(r).max()) for c, r in zip(covs, ref))
    PP.report(f"design interference_removal={interference_removal}", cov=err)
    assert err < DESIGN_REL
    if interference_removal:
        from scipy.linalg import eigh
        Cs = sum(ref)
        Cs = Cs + np.diag(np.mean(np.diag(Cs)) * np.ones(Cs.shape[0])) / 10
        want = np.stack([eigh(Cm, Cs - Cm)[1][:, -1] for Cm in ref], 1)
        want = want / np.linalg.norm(want, axis=0)
    else:
        want = np.stack([np.linalg.svd(Cm)[0][:, 0] for Cm in ref], 1)
    inner = np.abs(np.sum(np.conj(bf_mat) * want, axis=0))
    assert inner.min() >= 1 - 1e-5, inner.min()


# ---------------------------------------------------------------------------
# 4. against the existing paths
# ---------------------------------------------------------------------------
def test_agrees_with_hilbert_beamform_and_oracle():
    """On one context and input: power / DoA of micloc_hilbert_localize against micloc_hilbert_beamform (float32
    projections) and against the oracle's beamformer_apply on seeded one-second config-2 clips (front end 1e-4)."""
    from haghighatshoarmuir2024_b200 import _native as N
    from oracle import oracle as O
    g = dict(H.load("full_c2_b1"))
    T, B, M = 48_000, 3, 7
    eng = PP.engine(g, T)
    G = len(g["doa_list"])
    W = steering(M, G, 7)
    eng.set_hilbert_bf(W)
    x = H.synth_clips(g, B, T, seed=21, snrs_db=(0.0, 10.0, 20.0))[0]
    xd = PP.to_dev(x)
    out = eng.hilbert(xd)
    y = torch.empty((B, T, G, 2), dtype=torch.float32, device="cuda")
    pd = torch.empty((B, G), dtype=torch.float32, device="cuda")
    re, im = np.ascontiguousarray(W.real), np.ascontiguousarray(W.imag)
    N.check(N.lib().micloc_hilbert_beamform(eng._h, C.c_void_p(xd.data_ptr()), N.F32, B, T, re.ctypes.data_as(N._dp),
                                            im.ctypes.data_as(N._dp), G, C.c_void_p(y.data_ptr()),
                                            C.c_void_p(pd.data_ptr()), None, None))
    torch.cuda.synchronize()
    p, pdn = out["power"].cpu().numpy(), pd.cpu().numpy().astype(np.float64)
    e_dense = PP.rel_err(p, pdn)
    PP.check_doa(out["doa"].cpu().numpy(), pdn, DENSE_REL)
    po = np.stack([np.mean(np.abs(O.beamformer_apply(x[b], g["kernel"], g["ba_b"], g["ba_a"], W)) ** 2, axis=0)
                   for b in range(B)])
    e_or = PP.rel_err(p, po)
    PP.report("vs hilbert_beamform / oracle", dense=e_dense, oracle=e_or)
    assert e_dense < DENSE_REL
    assert e_or < 1e-4
    PP.check_doa(out["doa"].cpu().numpy(), po, 1e-4)


# ---------------------------------------------------------------------------
# 5. contract
# ---------------------------------------------------------------------------
def test_contract():
    """No steering matrix -> MICLOC_ERR_CONFIG for power / DoA (cov alone is fine); bad G, t_start outside [0, T) and
    the wrong number of microphones rejected; launches per call independent of B; two calls back to back on one
    stream without a synchronisation each return their own results; micloc_snn_run unchanged by set_hilbert_bf."""
    from haghighatshoarmuir2024_b200 import _native as N
    M, T, G = 7, 2000, 20
    g = PP.array_case(M, 4)
    eng = PP.engine(g, T)
    lib = N.lib()
    x = PP.clips(g, 600, T, seed=3)
    xd = PP.to_dev(x)
    doa = torch.empty(600, dtype=torch.int32, device="cuda")
    rc = lib.micloc_hilbert_localize(eng._h, C.c_void_p(xd.data_ptr()), N.F32, 600, T, 0, 1, None, None, None,
                                     C.c_void_p(doa.data_ptr()), None)
    assert rc == N.ERR_CONFIG
    eng.hilbert(xd, want=("cov",))
    ref = eng.run(xd[:8])
    ref = {k: v.clone() for k, v in ref.items() if v is not None}
    dummy = np.zeros((M, G))
    assert lib.micloc_hilbert_set_bf(eng._h, dummy.ctypes.data_as(N._dp), dummy.ctypes.data_as(N._dp), 0) == N.ERR_CONFIG
    with pytest.raises(ValueError):
        eng.set_hilbert_bf(np.zeros((M + 1, G), complex))
    W = steering(M, G, 9)
    eng.set_hilbert_bf(W)
    after = eng.run(xd[:8])
    torch.cuda.synchronize()
    for k, v in ref.items():
        assert torch.equal(after[k], v), k
    for bad in (T, -1):
        with pytest.raises(ValueError):
            eng.hilbert(xd[:2], t_start=bad)
    with pytest.raises(ValueError):
        eng.hilbert(PP.to_dev(PP.clips(PP.array_case(M + 1, 4), 2, T, seed=1)))
    counts = []
    for B in (5, 600):
        n0 = lib.micloc_launch_count()
        eng.hilbert(xd[:B])
        counts.append(lib.micloc_launch_count() - n0)
    assert counts[0] == counts[1] == 3, counts
    first = eng.hilbert(xd[:300], want=("power", "doa", "cov"))
    second = eng.hilbert(xd[300:], want=("power", "doa", "cov"))
    torch.cuda.synchronize()
    one = eng.hilbert(xd, want=("power", "doa", "cov"))
    torch.cuda.synchronize()
    for k in ("power", "doa", "cov"):
        assert torch.equal(torch.cat([first[k], second[k]]), one[k]), k


# ---------------------------------------------------------------------------
# 6. Monte-Carlo sweep, both arms on the same clips
# ---------------------------------------------------------------------------
def test_snr_sweep_hilbert_arm():
    """SnrSweep.run_band_hilbert on synthesised clips: its histogram sums to B, and at 20 dB both arms find the DoA
    within a few grid steps."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    from haghighatshoarmuir2024_b200.montecarlo import BandSetup, SnrSweep
    g = H.load("full_c2_b1")
    fs, T, B = float(g["fs"]), 48_000, 64
    doa_list = g["doa_list"]
    band = list(g["band"])
    bf = Beamformer(CenterCircularArray(4.5e-2, 7), float(g["kernel_duration"]), band, fs=fs)
    bf.verbose = False
    t = np.arange(4800) / fs
    bf_h, _ = bf.design_from_template((t, np.sin(2 * np.pi * band[1] * t)), doa_list)
    sweep = SnrSweep([BandSetup(band=band, tau=float(g["tau"]), bf_mat=g["bf_mat"], bf_hilbert=bf_h)],
                     g["r_vec"], g["theta_vec"], fs, float(g["kernel_duration"]), T)
    audio, doa_true, _ = sweep.synthesize(0, B, seed=4, snr_db_grid=[20.0])
    hist = torch.zeros(len(doa_list), dtype=torch.int64, device="cuda")
    hb = sweep.run_band_hilbert(0, audio, hist=hist)
    snn = sweep.run_band(0, audio)
    torch.cuda.synchronize()
    assert int(hist.sum()) == B
    step = doa_list[1] - doa_list[0]
    for out in (hb, snn):
        err = sweep.doa_error(out["doa"].cpu().numpy(), doa_true, doa_list)
        assert np.median(err) <= 3 * step, np.median(err)
