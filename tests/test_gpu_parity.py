"""Parity of the CUDA hot path (through the C-ABI) with the CPU oracle and with the
golden vectors of the real reference.  Needs a B200: run with -m gpu.

Tolerances are the ones BASELINE.json's north_star states:
  STHT output <= 1e-4 relative; spike time+sign agreement >= 99.9 %;
  identical DoA argmax on >= 99.5 % of frames (a frame = one clip).
"""
import numpy as np
import pytest
import torch
from scipy.signal import lfilter

import helpers as H
from oracle import oracle as O

pytestmark = pytest.mark.gpu

STHT_TOL = 1e-4
SPIKE_AGREE = 0.999
DOA_AGREE = 0.995


def engine_for(g, T=None):
    from haghighatshoarmuir2024_b200.engine import SnnEngine
    return SnnEngine(H.chain_spec(g, T), g["bf_mat"], device=0)


def to_dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


# ---------------------------------------------------------------------------
# golden vectors of the reference, stage by stage (staged kernels + taps)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", H.SNN_CASES)
def test_staged_taps_match_reference_golden(name):
    g = H.load(name)
    eng = engine_for(g)
    out = eng.run_taps(to_dev(g["x"]))
    torch.cuda.synchronize()
    rows = g["rows"]
    q = out["q"][0].cpu().numpy(); z = out["z"][0].cpu().numpy()
    assert H.rel_err(q[rows], g["q_rows"]) < STHT_TOL
    assert H.rel_err(z[rows], g["z_rows"]) < STHT_TOL
    spikes = out["spikes"][0].cpu().numpy()
    assert H.spike_agreement(spikes, g["spikes"]) >= SPIKE_AGREE
    assert int(out["flags"][0]) == 0
    # downstream of the spikes, always: the float64 alpha FIR of this call's own spikes (membrane, float32 recursion),
    # the float64 projection / power of this call's own membrane (k_dense, Gram + power)
    s = eng.spec
    n = np.arange(s.neuron_len)
    v64 = lfilter(s.neuron_scale * n * s.neuron_decay ** n, [1.0], spikes.astype(np.float64), axis=0)
    vm = out["vmem"][0].cpu().numpy().astype(np.float64)
    assert H.rel_err(vm, v64) < 1e-5
    y64 = vm @ g["bf_mat"]
    assert H.rel_err(out["y"][0].cpu().numpy(), y64) < 5e-6
    # (float64 Gram below 16 microphones, float32 tiles at 16, fp16 hi/lo tensor-core tiles at 64: measured 4.4e-6)
    assert H.rel_err(out["power"][0].cpu().numpy(), np.mean(y64 ** 2, axis=0)) < (2e-6 if eng.M < 64 else 6e-5)
    # and the reference's own values where the spikes are the reference's
    if np.array_equal(spikes, g["spikes"]):
        assert H.rel_err(out["vmem"][0].cpu().numpy()[rows], g["vmem_rows"]) < 1e-4
        assert H.rel_err(out["y"][0].cpu().numpy()[rows], g["y_rows"]) < 1e-4
        assert H.rel_err(out["power"][0].cpu().numpy(), g["power"]) < 1e-4
    assert int(out["doa"][0]) == int(g["doa"])


@pytest.mark.parametrize("variant", ["tc", "ffma"])
@pytest.mark.parametrize("name", H.SNN_CASES)
def test_fused_matches_reference_golden(name, variant, monkeypatch):
    g = H.load(name)
    eng = engine_for(g)
    if eng.M > 8:
        pytest.skip("the fused kernels cover up to 8 microphones; larger arrays take the tiled path")
    use_variant(monkeypatch, variant)
    out = eng.run(to_dev(g["x"]), want_spikes=True, fused=True)
    torch.cuda.synchronize()
    spikes = out["spikes"][0].cpu().numpy()
    assert H.spike_agreement(spikes, g["spikes"]) >= SPIKE_AGREE
    assert int(out["flags"][0]) == 0
    if np.array_equal(spikes, g["spikes"]):
        assert H.rel_err(out["power"][0].cpu().numpy(), g["power"]) < 1e-4
    assert int(out["doa"][0]) == int(g["doa"])


@pytest.mark.parametrize("name", H.FULL_CASES)
def test_one_second_clips_match_reference_golden(name, monkeypatch):
    """T = 48 000 goldens of the reference itself (configs[0] and one clip per band of configs[1]): staged taps and
    both fused kernels.  Pins the T-dependent neuron normalisation and a whole second of spikes on the device."""
    g = H.load(name)
    eng = engine_for(g)
    x = to_dev(g["x"])                                  # int16 PCM, the same integers the reference saw
    st = eng.run_taps(x, want=("q", "spikes", "vmem", "power", "doa"))
    torch.cuda.synchronize()
    rows = g["rows"]
    assert H.rel_err(st["q"][0].cpu().numpy()[rows], g["q_rows"]) < STHT_TOL
    sp = st["spikes"][0].cpu().numpy()
    assert H.spike_agreement(sp, g["spikes"]) >= SPIKE_AGREE
    # membrane rows away from the (few) differing spikes carry the kernel's normalisation: median relative error
    vm = st["vmem"][0].cpu().numpy()[rows]
    scale = np.abs(g["vmem_rows"]).max()
    assert np.median(np.abs(vm - g["vmem_rows"])) / scale < 1e-6
    assert H.rel_err(st["power"][0].cpu().numpy(), g["power"]) < 2e-3
    assert int(st["doa"][0]) == int(g["doa"])
    for variant in VARIANTS:
        use_variant(monkeypatch, variant)
        fu = eng.run(x, want_spikes=True, fused=True)
        torch.cuda.synchronize()
        assert int(fu["flags"][0]) == 0
        assert H.spike_agreement(fu["spikes"][0].cpu().numpy(), g["spikes"]) >= SPIKE_AGREE, variant
        assert H.rel_err(fu["power"][0].cpu().numpy(), g["power"]) < 2e-3, variant
        assert int(fu["doa"][0]) == int(g["doa"]), variant


VARIANTS = ["tc", "ffma"]     # fused kernels: STHT on the tensor cores (default) / on the FP32 FMA pipe


def use_variant(monkeypatch, variant):
    if variant == "ffma":
        monkeypatch.setenv("MICLOC_FUSED_FIR", "ffma")
    else:
        monkeypatch.delenv("MICLOC_FUSED_FIR", raising=False)


def same_spikes(fused, staged, variant, floor=SPIKE_AGREE):
    """The FFMA kernel repeats the staged kernels' float32 arithmetic in the same order (identical spikes); the
    tensor-core kernel sums the STHT in another order (hi/lo fp16 products, float32 accumulation) and is held to
    the north-star tolerance."""
    if variant == "ffma":
        return torch.equal(fused, staged)
    return H.spike_agreement(fused.cpu().numpy(), staged.cpu().numpy()) >= floor


def _sub_array(g, mics):
    """The golden case restricted to a subset of its microphones (rows of bf_mat follow: in-phase | quadrature)."""
    M = g["x"].shape[1]
    mics = np.asarray(mics)
    g2 = dict(g)
    g2["x"] = np.ascontiguousarray(g["x"][:, mics])
    g2["r_vec"], g2["theta_vec"] = g["r_vec"][mics], g["theta_vec"][mics]
    g2["bf_mat"] = np.ascontiguousarray(g["bf_mat"][np.concatenate([mics, M + mics])])
    return g2


@pytest.mark.parametrize("mics,variant", [((0, 2, 3, 5), "tc"), ((1, 2, 3, 4, 6), "tc"), ((0, 1, 2, 3, 4, 5), "tc"), ((3,), "tc"),
                                          ((0, 2, 3, 5), "ffma"), ((0, 1, 2, 3, 4, 5), "ffma"), ((3,), "ffma")])
def test_smaller_arrays_generic_microphone_count(mics, variant, monkeypatch):
    """Arrays of 1...6 microphones take the fused kernels' generic-M instantiation: fused vs staged vs oracle."""
    g = _sub_array(H.load("snn_c1_bipolar"), mics)
    T, B = 4000, 12
    x, _ = H.synth_clips(g, B, T, seed=77 + len(mics))
    eng = engine_for(g, T)
    st = eng.run(to_dev(x), want_spikes=True, fused=False)
    use_variant(monkeypatch, variant)
    fu = eng.run(to_dev(x), want_spikes=True, fused=True)
    torch.cuda.synchronize()
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / float(g["fs"]), float(g["tau"]), float(g["tau"]))
    ref = O.snn_run_batch(cfg, x, nthreads=4, want_spikes=True)
    assert same_spikes(fu["spikes"], st["spikes"], variant)
    assert H.spike_agreement(fu["spikes"].cpu().numpy(), ref["spikes"]) >= SPIKE_AGREE
    assert (fu["doa"].cpu().numpy() == ref["doa"]).mean() >= 0.9      # 12 clips: one near-tie may flip
    assert H.rel_err(fu["power"].cpu().numpy(), st["power"].cpu().numpy()) < (1e-5 if variant == "ffma" else 2e-3)
    assert int(fu["flags"].sum()) == 0


# ---------------------------------------------------------------------------
# batches against the oracle: fused and staged agree within the reference tolerance with each other
# (their float32 Gram sums run on different units) and with the oracle
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name,T,int16", [("snn_c1_bipolar", 4800, False), ("snn_c1_unipolar", 3000, False),
                                          ("snn_band2_sine", 4801, True), ("snn_band3_i16", 1000, True),
                                          ("snn_k20ms", 2500, False)])
def test_batch_fused_vs_staged_vs_oracle(name, T, int16, variant, monkeypatch):
    g = H.load(name)
    B = 48
    x, _ = H.synth_clips(g, B, T, seed=100 + T, int16=int16)
    eng = engine_for(g, T)
    xd = to_dev(x)
    st = eng.run(xd, want_spikes=True, fused=False)
    use_variant(monkeypatch, variant)
    fu = eng.run(xd, want_spikes=True, fused=True)
    torch.cuda.synchronize()
    # FFMA kernel: same STHT / band-pass / RZCC arithmetic in the same order as the staged kernels (identical
    # spikes; the Gram sums differ: fp16 hi/lo tensor-core products vs FP64)
    assert same_spikes(fu["spikes"], st["spikes"], variant)
    assert (st["doa"] == fu["doa"]).float().mean().item() >= DOA_AGREE
    assert H.rel_err(fu["power"].cpu().numpy(), st["power"].cpu().numpy()) < (1e-5 if variant == "ffma" else 2e-3)
    cfg = H.oracle_cfg(g)
    fs = float(g["fs"]); tau = float(g["tau"])
    cfg.nir = O.neuron_kernel(np.arange(T) / fs, tau, tau)
    ref = O.snn_run_batch(cfg, x, nthreads=8, want_spikes=True)
    sp = fu["spikes"].cpu().numpy()
    assert H.spike_agreement(sp, ref["spikes"]) >= SPIKE_AGREE
    same = (fu["doa"].cpu().numpy() == ref["doa"]).mean()
    assert same >= DOA_AGREE, f"DoA agreement {same}"
    assert int(fu["flags"].sum()) == 0


def test_full_size_clip_config1():
    """Config 1 size (1 s, 48 kHz, 7 mics, G=64): one clip against the oracle + properties."""
    g = H.load("snn_c1_bipolar")
    T = 48000
    x, _ = H.synth_clips(g, 4, T, seed=7, snrs_db=(20.0,))
    eng = engine_for(g, T)
    out = eng.run(to_dev(x), want_spikes=True, fused=True)
    tap = eng.run_taps(to_dev(x[:1]), want=("q",))
    torch.cuda.synchronize()
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / 48000.0, float(g["tau"]), float(g["tau"]))
    ref = O.snn_apply(cfg, x[0].astype(np.float64), want=("q", "spikes", "power"))
    assert H.rel_err(tap["q"][0].cpu().numpy(), ref["q"]) < STHT_TOL
    assert H.spike_agreement(out["spikes"][0].cpu().numpy(), ref["spikes"]) >= SPIKE_AGREE
    assert int(out["doa"][0]) == ref["doa"]
    # size-independent properties: scale invariance of spikes/DoA, linearity of the STHT
    out2 = eng.run(to_dev(x * np.float32(4.0)), want_spikes=True, fused=True)
    assert torch.equal(out2["spikes"], out["spikes"]) and torch.equal(out2["doa"], out["doa"])
    s = out["spikes"][0].cpu().numpy()
    assert not s[0].any() and not s[-1].any()          # first / last sample never spike
    for c in range(s.shape[1]):                        # kept spikes of one sign are >= w apart
        for sign in (1, -1):
            pos = np.flatnonzero(s[:, c] == sign)
            assert pos.size < 2 or np.diff(pos).min() >= int(g["robust_width"])


def test_full_size_config2_three_bands_449_grid():
    """Config 2 size (bench.py's workload): 1 s clips, three bands, G = 449, 11 SNRs from -10 to 20 dB -- the fused
    kernel against the oracle on 192 clips per band: spike agreement, DoA match rate, and the DoA histogram kernel."""
    import sys
    sys.path.insert(0, H.ROOT)
    import bench as Bn
    from haghighatshoarmuir2024_b200.montecarlo import BandSetup, SnrSweep
    d, bands = Bn.load_workload()
    setups = [BandSetup(band=bands[i], tau=float(d[f"tau_{i}"]), bf_mat=d[f"bf_{i}"]) for i in range(len(bands))]
    sweep = SnrSweep(setups, d["r_vec"], d["theta_vec"], Bn.FS, float(d["kernel_duration"]), Bn.T_CLIP, device=0)
    cfgs = Bn.oracle_cfgs(d, bands)
    n = 192
    match = total = 0
    for i in range(len(bands)):
        x = Bn.host_clips(d, i, bands, n, seed=500 + i)
        hist = torch.zeros(sweep.G, dtype=torch.int64, device="cuda")
        out = sweep.run_band(i, to_dev(x), want_spikes=True, want_power=True, hist=hist)
        torch.cuda.synchronize()
        ref = O.snn_run_batch(cfgs[i], x, nthreads=8, want_spikes=True)
        assert H.spike_agreement(out["spikes"].cpu().numpy(), ref["spikes"]) >= SPIKE_AGREE, i
        doa = out["doa"].cpu().numpy()
        match += int((doa == ref["doa"]).sum()); total += n
        assert np.array_equal(hist.cpu().numpy(), np.bincount(doa, minlength=sweep.G)), i
        assert int(out["flags"].sum()) == 0
    assert match / total >= DOA_AGREE, f"DoA match rate {match}/{total}"


def test_full_size_config4_multi_source_360_grid():
    """Config 4 size: 1 s clips with two simultaneous sources, G = 360, fused kernel vs oracle."""
    g = H.load("snn_c4_multi")
    T = 48000
    rng = np.random.default_rng(41)
    fs = float(g["fs"]); t = np.arange(T) / fs
    from scipy.signal import butter, lfilter
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    geo = ArrayGeometry(g["r_vec"], g["theta_vec"])
    b_, a_ = butter(2, g["band"], btype="bandpass", fs=fs)
    xs = []
    for i in range(3):
        src = lfilter(b_, a_, lfilter([1.0], [1.0, -0.95], rng.standard_normal(T)))
        x = 0.0
        for doa in (np.pi / 3, -np.pi / 3 + 0.2 * i):          # multiple_targets_snn.py:87-159: delays added, np.interp
            x = x + np.interp((t[:, None] + geo.delays_batch(np.full(T, doa))).ravel(), t, src).reshape(T, -1)
        xs.append(x + 0.05 * np.std(x) * rng.standard_normal(x.shape))
    x = np.stack(xs).astype(np.float32)
    eng = engine_for(g, T)
    out = eng.run(to_dev(x), want_spikes=True, fused=True)
    st = eng.run(to_dev(x), want_spikes=True, fused=False)
    assert same_spikes(out["spikes"], st["spikes"], "tc") and torch.equal(out["doa"], st["doa"])
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(t, float(g["tau"]), float(g["tau"]))
    ref = O.snn_run_batch(cfg, x, nthreads=3, want_spikes=True)
    assert H.spike_agreement(out["spikes"].cpu().numpy(), ref["spikes"]) >= SPIKE_AGREE
    assert np.array_equal(out["doa"].cpu().numpy(), ref["doa"])
    assert H.rel_err(out["power"].cpu().numpy(), ref["power"]) < 2e-3
    assert int(out["flags"].sum()) == 0


@pytest.mark.parametrize("name", ["snn_c5_random64", "snn_c5_linear64"])
def test_full_size_config5_64_mics_10s_512_grid(name):
    """Config 5 size: one 10 s clip (T = 480 000) on the 64-microphone arrays, G = 512, against the oracle.  Few long
    clips take the time-segmented kernels (k_chain_blk / k_neuron_seg / k_gram_slab)."""
    import time
    g = H.load(name)
    T = 480_000
    x, _ = H.synth_clips(g, 1, T, seed=51, snrs_db=(10.0,))
    eng = engine_for(g, T)
    xd = to_dev(x)
    out = eng.run(xd, want_spikes=True, fused=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = eng.run(xd, want_spikes=True, fused=False)
    torch.cuda.synchronize()
    ms = 1e3 * (time.perf_counter() - t0)
    print(f"config 5 ({name}): {ms:.1f} ms per 10 s clip")
    assert ms < 100.0                                     # (tens of seconds per clip before the segmented kernels)
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / float(g["fs"]), float(g["tau"]), float(g["tau"]))
    ref = O.snn_run_batch(cfg, x, nthreads=1, want_spikes=True)
    assert H.spike_agreement(out["spikes"].cpu().numpy(), ref["spikes"]) >= SPIKE_AGREE
    assert int(out["doa"][0]) == int(ref["doa"][0])
    assert H.rel_err(out["power"].cpu().numpy(), ref["power"]) < 2e-3
    assert int(out["flags"].sum()) == 0


def test_time_segmented_kernels_equal_the_sequential_ones(monkeypatch):
    """Few long clips: (clip, channel, time segment) chains with warm-up against one chain per (clip, channel)."""
    for name, B, T in (("snn_c5_random64", 1, 100_000), ("snn_c1_bipolar", 3, 70_001), ("snn_c1_unipolar", 2, 48_000)):
        g = H.load(name)
        x, _ = H.synth_clips(g, B, T, seed=7, snrs_db=(0.0, 15.0))
        x[-1, T // 3: T // 3 + 9000] = 0                                # a stretch of digital silence inside one clip
        eng = engine_for(g, T)
        xd = to_dev(x)
        monkeypatch.delenv("MICLOC_NO_SEGMENTS", raising=False)
        seg = eng.run_taps(xd, want=("spikes", "vmem", "power", "doa"))
        monkeypatch.setenv("MICLOC_NO_SEGMENTS", "1")
        one = eng.run_taps(xd, want=("spikes", "vmem", "power", "doa"))
        torch.cuda.synchronize()
        assert H.spike_agreement(seg["spikes"].cpu().numpy(), one["spikes"].cpu().numpy()) >= 0.9999, name
        assert H.rel_err(seg["power"].cpu().numpy(), one["power"].cpu().numpy()) < 1e-3
        assert torch.equal(seg["doa"], one["doa"])
        assert torch.equal(seg["flags"], one["flags"])


def test_wide_array_tensor_core_gram_and_sliced_power_equal_the_float64_sum(monkeypatch):
    """64 microphones (128 channels): k_gram_tc (fp16 hi/lo mma.sync) + k_power_wide against the float32 tiled product and
    against the plain float64 sum with one thread per DoA; ragged T (last slab and last k step partly empty)."""
    g = H.load("snn_c5_linear64")
    for B, T in ((2, 20_011), (1, 3_000)):
        x, _ = H.synth_clips(g, B, T, seed=11, snrs_db=(5.0,))
        eng = engine_for(g, T)
        xd = to_dev(x)
        for k in ("MICLOC_GRAM_FP32", "MICLOC_POWER_NARROW", "MICLOC_NO_SEGMENTS"):
            monkeypatch.delenv(k, raising=False)
        tc = eng.run_taps(xd, want=("power", "doa"))
        monkeypatch.setenv("MICLOC_GRAM_FP32", "1")
        monkeypatch.setenv("MICLOC_POWER_NARROW", "1")
        f32 = eng.run_taps(xd, want=("power", "doa"))
        monkeypatch.setenv("MICLOC_NO_SEGMENTS", "1")                    # float64 Gram, one thread per matrix element
        f64 = eng.run_taps(xd, want=("power", "doa"))
        torch.cuda.synchronize()
        p64 = f64["power"].cpu().numpy()
        assert H.rel_err(tc["power"].cpu().numpy(), p64) < 1e-5, (B, T)
        assert H.rel_err(f32["power"].cpu().numpy(), p64) < 1e-5, (B, T)
        assert torch.equal(tc["doa"], f64["doa"]) and torch.equal(f32["doa"], f64["doa"])


@pytest.mark.parametrize("name", ["snn_c5_linear64", "snn_linear16"])
def test_wide_array_tensor_core_stht_equals_the_fp32_fir(name, monkeypatch):
    """M > 8: k_stht_tc (polyphase Toeplitz product, fp16 hi/lo mma.sync) against the float32 FIR kernel and the
    float64 oracle; float32 and int16 clips, ragged T (partial tiles, odd length), loud and quiet clips in one batch."""
    g = H.load(name)
    M = g["x"].shape[1]
    for T, int16 in ((5_001, False), (777, False), (4_096, True)):
        x, _ = H.synth_clips(g, 3, T, seed=T)
        x[1] *= 1e-3                                                     # per-tile scaling: a quiet clip next to a loud one
        x[2, : T // 2] = 0
        if int16:
            x = np.round(x / np.abs(x).max() * 30000).astype(np.int16)
        eng = engine_for(g, max(T, 1024))
        xd = to_dev(x)
        monkeypatch.delenv("MICLOC_STHT_FP32", raising=False)
        q_tc = eng.run_taps(xd, want=("q",))["q"].cpu().numpy()
        monkeypatch.setenv("MICLOC_STHT_FP32", "1")
        q_32 = eng.run_taps(xd, want=("q",))["q"].cpu().numpy()
        monkeypatch.delenv("MICLOC_STHT_FP32", raising=False)
        h = np.asarray(g["kernel"], np.float64)
        for bi in range(3):
            ref = np.stack([np.convolve(x[bi, :, m].astype(np.float64), h)[:T] for m in (0, M // 2, M - 1)], axis=1)
            got = q_tc[bi][:, [0, M // 2, M - 1]]
            assert H.rel_err(got, ref) < 1e-5, (T, int16, bi)
            assert H.rel_err(q_32[bi][:, [0, M // 2, M - 1]], ref) < 1e-5
        assert np.isfinite(q_tc).all()


def test_stht_linearity_and_zero_input():
    g = H.load("snn_c1_bipolar")
    eng = engine_for(g, 2048)
    rng = np.random.default_rng(0)
    a = rng.standard_normal((1, 2048, 7)).astype(np.float32)
    b = rng.standard_normal((1, 2048, 7)).astype(np.float32)
    qa = eng.run_taps(to_dev(a), want=("q",))["q"]; qb = eng.run_taps(to_dev(b), want=("q",))["q"]
    qab = eng.run_taps(to_dev(a + b), want=("q",))["q"]
    assert H.rel_err((qa + qb).cpu().numpy(), qab.cpu().numpy()) < 1e-5
    zero = eng.run(to_dev(np.zeros((2, 2048, 7), np.float32)), want_spikes=True, fused=True)
    assert int(zero["spikes"].abs().sum()) == 0 and int(zero["doa"][0]) == 0      # all-equal power -> first index


@pytest.mark.parametrize("variant", VARIANTS)
def test_ragged_and_tiny_clips(variant, monkeypatch):
    g = H.load("snn_c1_bipolar")
    cfg = H.oracle_cfg(g)
    for T in (1, 2, 3, 17, 127, 128, 129, 255, 256, 257, 481, 1023):
        x, _ = H.synth_clips(g, 3, T, seed=T)
        eng = engine_for(g, max(T, 64))
        monkeypatch.delenv("MICLOC_FUSED_FIR", raising=False)
        st = eng.run(to_dev(x), want_spikes=True, fused=False)
        use_variant(monkeypatch, variant)
        fu = eng.run(to_dev(x), want_spikes=True, fused=True)
        torch.cuda.synchronize()
        assert same_spikes(fu["spikes"], st["spikes"], variant, floor=0.99), T
        ref = O.snn_run_batch(cfg, x, nthreads=1, want_spikes=True)
        assert H.spike_agreement(fu["spikes"].cpu().numpy(), ref["spikes"]) >= 0.99, T


def test_shape_errors_raise_valueerror():
    g = H.load("snn_c1_bipolar")
    eng = engine_for(g)
    with pytest.raises(ValueError):
        eng.run(torch.zeros((1, 100, 6), device="cuda"))
    with pytest.raises(ValueError):
        eng.run(torch.zeros((1, 100, 7), device="cuda", dtype=torch.float64))


def test_run_host_end_to_end_equals_device_path():
    g = H.load("snn_band3_i16")
    x, _ = H.synth_clips(g, 40, 2400, seed=5, int16=True)
    eng = engine_for(g, 2400)
    dev = eng.run(to_dev(x), want_spikes=True, fused=True)
    torch.cuda.synchronize()
    host = eng.run_host(torch.from_numpy(x).pin_memory(), want_spikes=True, fused=True)
    assert np.array_equal(host["doa"].numpy(), dev["doa"].cpu().numpy())
    assert np.array_equal(host["spikes"].numpy(), dev["spikes"].cpu().numpy())
    np.testing.assert_array_equal(host["power"].numpy(), dev["power"].cpu().numpy())


def test_run_host_overlapping_chunks_equal_device_path(monkeypatch):
    """Several chunks in flight on the two staging streams (the fused kernel's dynamic clip-pair
    counter is per stream) must give what one device launch gives."""
    g = H.load("snn_c1_bipolar")
    x, _ = H.synth_clips(g, 700, 1200, seed=9)
    eng = engine_for(g, 1200)
    dev = eng.run(to_dev(x), want_spikes=True, fused=True)
    torch.cuda.synchronize()
    monkeypatch.setenv("MICLOC_HOST_CHUNK_CLIPS", "90")
    for _ in range(3):
        host = eng.run_host(torch.from_numpy(x).pin_memory(), want_spikes=True, fused=True)
        assert np.array_equal(host["doa"].numpy(), dev["doa"].cpu().numpy())
        assert np.array_equal(host["spikes"].numpy(), dev["spikes"].cpu().numpy())


# ---------------------------------------------------------------------------
# stand-alone stages
# ---------------------------------------------------------------------------
def test_rzcc_encoder_bit_exact_on_reference_golden():
    from haghighatshoarmuir2024_b200.spike_encoder import ZeroCrossingSpikeEncoder
    g = H.load("rzcc")
    n = 0
    for key in g:
        if not key.startswith("spk_"):
            continue
        _, sname, w, b = key.split("_")
        enc = ZeroCrossingSpikeEncoder(fs=48000, robust_width=int(w[1:]), bipolar=bool(int(b[1:])))
        got = enc.evolve(g["sig_" + sname])
        assert got.dtype == np.float64 and np.array_equal(got.astype(np.int8), g[key]), key
        n += 1
    assert n == 32


def test_rzcc_encoder_white_noise_matches_oracle_and_rejects_bad_width():
    from haghighatshoarmuir2024_b200.spike_encoder import ZeroCrossingSpikeEncoder
    rng = np.random.default_rng(9)
    x = rng.standard_normal((20000, 4))
    for w in (2, 12, 40):
        got = ZeroCrossingSpikeEncoder(48000, w, True).evolve(x)
        assert np.array_equal(got, O.rzcc(x, w, True))
    with pytest.raises(ValueError):
        ZeroCrossingSpikeEncoder(48000, 0, True).evolve(x)


def test_hilbert_beamformer_matches_reference_golden():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    g = H.load("beamformer")
    bf = Beamformer(CenterCircularArray(4.5e-2, 7), 10e-3, list(g["band"]), fs=float(g["fs"]))
    y = bf.apply_to_signal(g["bf_mat"], g["x"].astype(np.float64))
    assert y.dtype == np.complex128 and y.shape == (g["x"].shape[0], g["bf_mat"].shape[1])
    assert H.rel_err(y[g["rows"]], g["y_rows"]) < 1e-4
    power = np.mean(np.abs(y) ** 2, axis=0)
    assert int(np.argmax(power)) == int(g["doa"])
    with pytest.raises(ValueError):
        bf.apply_to_signal(g["bf_mat"], np.zeros((100, 6)))


# ---------------------------------------------------------------------------
# drop-in classes
# ---------------------------------------------------------------------------
def test_snn_beamformer_dropin_apply_and_design():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
    g = H.load("snn_c1_bipolar")
    tau = float(g["tau"])
    beamf = SNNBeamformer(CenterCircularArray(4.5e-2, 7), float(g["kernel_duration"]), list(g["band"]),
                          np.array([tau, tau]), bipolar_spikes=True, fs=float(g["fs"]))
    beamf.verbose = False
    assert beamf.kernel_length == len(g["kernel"]) and beamf.spk_encoder.robust_width == int(g["robust_width"])
    np.testing.assert_allclose(beamf.kernel, g["kernel"], atol=1e-15)
    T = g["x"].shape[0]
    t = np.arange(T) / float(g["fs"])
    y = beamf.apply_to_signal(g["bf_mat"], (t, g["x"].astype(np.float64)))
    assert y.dtype == np.float64 and y.shape == (T, g["bf_mat"].shape[1])
    power = np.mean(np.abs(y) ** 2, axis=0)
    assert int(np.argmax(power)) == int(g["doa"])
    with pytest.raises(ValueError):
        beamf.apply_to_signal(g["bf_mat"], (t, np.zeros((T, 5))))
    # design_from_template against the reference's matrix (columns up to a global sign)
    bf = beamf.design_from_template((t, g["template"]), g["doa_list"])
    assert bf.shape == g["bf_mat"].shape
    M = 7                                             # columns are complex vectors up to a global phase
    u = bf[:M] + 1j * bf[M:]; ur = g["bf_mat"][:M] + 1j * g["bf_mat"][M:]
    d = np.abs(np.sum(u.conj() * ur, axis=0))
    assert d.min() > 0.999
    with pytest.raises(ValueError):
        SNNBeamformer(CenterCircularArray(4.5e-2, 7), 10e-3, [2000, 1000], np.array([tau, tau]))


def test_snn_beamformer_unipolar_design_matches_reference():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
    g = H.load("snn_c1_unipolar")
    tau = float(g["tau"])
    beamf = SNNBeamformer(CenterCircularArray(4.5e-2, 7), 10e-3, list(g["band"]), np.array([tau, tau]),
                          bipolar_spikes=False, fs=48000)
    beamf.verbose = False
    t = np.arange(g["x"].shape[0]) / 48000.0
    bf = beamf.design_from_template((t, g["template"]), g["doa_list"])
    d = np.abs(np.sum(bf * g["bf_mat"], axis=0))
    assert d.min() > 0.995


@pytest.mark.parametrize("variant", ["tc", "ffma"])
def test_rzcc_overflow_is_healed_by_the_library(variant, monkeypatch):
    """Digital silence inside a clip: the band-pass output is the filter's decaying tail.  Once it no longer moves the
    running sum (rzcc_flat: |z| < 2^-53 |sum|, the reference's float64 np.cumsum behaves the same way at its own
    scale) the float32 chains see a flat top; when the signal resumes, that flat top is longer than the fused kernel's
    streaming encoder follows (flags bit 0) and micloc_snn_refine / run_host / the staged entry points redo the clip
    with the unbounded float64 encoder.  Inside the silence the reference's spikes are decided by float64 values below
    the float32 range (1e-45 ... 1e-115), so the comparison with the oracle leaves the silent stretch out."""
    g = H.load("snn_c1_bipolar")
    T, B = 24_000, 6
    x, _ = H.synth_clips(g, B, T, seed=21, snrs_db=(10.0,))
    silent = {1: (3000, 15000), 3: (2000, 16000), 4: (9000, T)}
    for b, (s0, s1) in silent.items():
        x[b, s0:s1] = 0             # clips 1, 3: the signal resumes, on some channel with the opposite sign; 4: trailing
    eng = engine_for(g, T)
    xd = to_dev(x)
    taps = eng.run_taps(xd, want=("z", "spikes", "power", "doa"))
    torch.cuda.synchronize()
    assert int(taps["flags"].sum()) == 0 and eng.refined_count >= 2          # healed inside the staged call
    z = taps["z"].cpu().numpy()
    z[np.abs(z) < np.finfo(np.float32).tiny] = 0                              # (the heal path drops denormals)
    for b in (1, 3):
        want = O.rzcc(z[b].astype(np.float64), float(eng.spec.robust_width), True)
        assert np.array_equal(taps["spikes"][b].cpu().numpy(), want), b
    assert int(taps["spikes"][4, 16000:].abs().sum()) == 0                    # silent in silence, not a denormal limit cycle
    use_variant(monkeypatch, variant)
    raw = eng.run(xd, want_spikes=True, fused=True, refine=False)
    torch.cuda.synchronize()
    flagged = (raw["flags"].cpu().numpy() & 1).astype(bool)
    assert flagged[1] and flagged[3] and not flagged[0] and not flagged[4]
    assert int(raw["spikes"][4, 16000:].abs().sum()) == 0
    n = eng.refine(xd, raw)
    torch.cuda.synchronize()
    assert n == int(flagged.sum()) and int(raw["flags"].sum()) == 0
    for b in np.nonzero(flagged)[0]:
        assert torch.equal(raw["spikes"][b], taps["spikes"][b])
        assert H.rel_err(raw["power"][b].cpu().numpy(), taps["power"][b].cpu().numpy()) < 1e-5
        assert int(raw["doa"][b]) == int(taps["doa"][b])
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / float(g["fs"]), float(g["tau"]), float(g["tau"]))
    ref = O.snn_run_batch(cfg, x, nthreads=B, want_spikes=True)
    got = raw["spikes"].cpu().numpy()
    for b in range(B):
        keep = np.ones(T, bool)
        if b in silent:
            keep[silent[b][0] + 1000: min(T, silent[b][1] + 600)] = False     # tail beyond float32 + the restart transient
        assert H.spike_agreement(got[b][keep], ref["spikes"][b][keep]) >= SPIKE_AGREE, b
    live = [b for b in range(B) if b not in silent]
    assert np.array_equal(raw["doa"].cpu().numpy()[live], ref["doa"][live])
    auto = eng.run(xd, want_spikes=True, fused=True)                         # refine=True is the default
    assert int(auto["flags"].sum()) == 0 and torch.equal(auto["spikes"], raw["spikes"])
    host = eng.run_host(torch.from_numpy(x).pin_memory(), want_spikes=True, fused=True)
    assert int(host["flags"].sum()) == 0
    assert torch.equal(host["spikes"], raw["spikes"].cpu()) and torch.equal(host["doa"], raw["doa"].cpu())
