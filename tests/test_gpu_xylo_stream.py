"""Xylo stream batches (micloc_xylo_streams_*): many continuous recordings through the exact front end and the integer
network, one push per frame tick.

Bar: bit for bit.  N pushed frames plus a flush give, for every slot, what XyloEngine.run(exact=True) and the CPU oracle
give on one clip of their concatenation (clips whose last K/2 samples are zero, where the causal in-phase delay equals
np.roll), whenever the slot's flags bit 0 is clear."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
from haghighatshoarmuir2024_b200 import _native as N
from oracle import oracle as O

FRAMES = (1, 31, 63, 64, 65, 448, 1000, 700, 1000, 628)       # 448 < D = 449 (w = 12); 1000 = max_frame_len
MAX_FRAME = 1000
T_TOTAL = sum(FRAMES)


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def zero_tail(x, g):
    x = np.array(x)
    x[:, -(len(g["kernel"]) // 2):] = 0
    return x


def stream_batch(eng, S, max_frame=MAX_FRAME, **kw):
    from haghighatshoarmuir2024_b200.xylo_snn_localization import XyloStreamBatch
    return XyloStreamBatch(eng, S, max_frame, **kw)


def run_stream(xsb, x, frames=FRAMES, peak_win=0):
    """Push x [S, T, ch] in `frames`, then flush.  Returns per-slot concatenated spikes_in / raster rows, summed counts,
    the per-call outputs and the flags of the last push and of the flush."""
    S = x.shape[0]
    sp = [[] for _ in range(S)]
    ra = [[] for _ in range(S)]
    counts = np.zeros((S, xsb.N), dtype=np.int64)
    calls, t = [], 0
    for n in list(frames) + [None]:
        if n is None:
            out = xsb.flush(want_spikes_in=True, want_raster=True, peak_win=peak_win)
        else:
            out = xsb.push(dev(x[:, t:t + n]), want_spikes_in=True, want_raster=True, peak_win=peak_win)
            t += n
        m = out["n_out"]
        si, r = out["spikes_in"].cpu().numpy(), out["raster"].cpu().numpy()
        c = out["counts"].cpu().numpy()
        for s in range(S):
            sp[s].append(si[s, :m[s]])
            ra[s].append(r[s, :m[s]])
        counts += c
        calls.append({k: (v.cpu().numpy() if torch.is_tensor(v) else v) for k, v in out.items()
                      if k not in ("spikes_in", "raster")})
    assert t == x.shape[1]
    return ([np.concatenate(a) for a in sp], [np.concatenate(a) for a in ra], counts, calls)


def signed(spikes_in, CT, bipolar):
    s = spikes_in.astype(np.int8)
    return s[..., :CT] - s[..., CT:] if bipolar else s


def check_against_clip(eng, x, got, cfg=None, fs=48000.0):
    """The stream's rows against the one-shot exact chain (and the oracle when cfg is given) on the same clips."""
    sp, ra, counts, calls = got
    ref = eng.run(dev(x), exact=True, want_spikes_in=True, want_raster=True)
    S, T = x.shape[:2]
    assert sum(c["n_out"] for c in calls).tolist() == [T] * S
    for s in range(S):
        assert np.array_equal(sp[s], ref["spikes_in"][s].cpu().numpy()), s
        assert np.array_equal(ra[s], ref["raster"][s].cpu().numpy()), s
    assert np.array_equal(counts, ref["counts"].cpu().numpy())
    assert int(calls[-1]["flags"].max()) & 1 == 0 and int(ref["flags"].sum()) == 0
    if cfg is not None:
        o = O.xylo_run_batch(cfg, np.ascontiguousarray(x), fs, win=0, nthreads=4, want_spikes=True)
        for s in range(S):
            assert np.array_equal(signed(sp[s], eng.CT, cfg.bipolar), o["spikes_signed"][s]), s
        assert np.array_equal(counts, o["counts"])


@pytest.mark.gpu
@pytest.mark.parametrize("name,int16", [("xylo_c3_bipolar", False), ("xylo_c3_bipolar", True),
                                        ("xylo_c3_unipolar", False), ("xylo_3band_o2", False)])
def test_stream_equals_one_shot_clip_and_oracle(name, int16):
    g = H.load(name)
    net = H.xylo_network(g)
    eng = H.xylo_engine(g, net)
    x = zero_tail(H.xylo_synth_clips(g, 5, T_TOTAL, seed=41, int16=int16), g)
    xsb = stream_batch(eng, 5)
    assert xsb.latency == 31 * 11 + 12 + 96
    check_against_clip(eng, x, run_stream(xsb, x), H.xylo_oracle_cfg(g, net))


@pytest.mark.gpu
def test_int32_wav_frames_take_the_float64_sample_path():
    """T x 8 int32 frames with samples up to 2^30 (not float32-exact) and a junk 8th channel, against the oracle's
    float64 encoder and network on the concatenation."""
    g = H.load("xylo_c3_bipolar")
    net = H.xylo_network(g)
    eng = H.xylo_engine(g, net)
    cfg = H.xylo_oracle_cfg(g, net)
    rng = np.random.default_rng(3)
    x = H.xylo_synth_clips(g, 3, T_TOTAL, seed=9).astype(np.float64)
    x = np.round(x / np.abs(x).max() * (2 ** 30 - 1)) + rng.integers(-7, 8, size=x.shape)
    x = zero_tail(x, g).astype(np.int32)
    assert np.any(x.astype(np.float32).astype(np.int64) != x)          # float32 would round these samples
    wav = np.concatenate([x, rng.integers(-2 ** 31, 2 ** 31 - 1, size=(3, T_TOTAL, 1), dtype=np.int64).astype(np.int32)], 2)
    sp, ra, counts, calls = run_stream(stream_batch(eng, 3), wav)
    for s in range(3):
        ref_in, _ = O.xylo_encode(cfg, x[s].astype(np.float64))
        assert np.array_equal(sp[s], ref_in), s
        raster, cnt = O.xylo_lif(cfg, ref_in)
        assert np.array_equal(ra[s], raster) and np.array_equal(counts[s], cnt), s
    assert int(calls[-1]["flags"].max()) == 0


@pytest.mark.gpu
def test_per_call_counts_doa_rate_and_estimators():
    """counts / doa / doa_peak of every call against the oracle raster over that call's rows; rate, periodic_ml and
    trimmed_periodic_ml against Demo.extract_rate / estimate_doa_from_rate on the host, including the trimmed
    estimator's IndexError case (NaN + flags bit 1)."""
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.xylo_snn_localization import Demo, signal_from_template
    g = H.load("xylo_c3_bipolar")
    geo = ArrayGeometry(g["r_vec"], g["theta_vec"])
    demo = Demo(geometry=geo, freq_bands=g["bands"], doa_list=g["doa_list"], recording_duration=0.05,
                kernel_duration=float(g["kernel_duration"]), bipolar_spikes=True, fs=float(g["fs"]),
                bf_mats=list(g["bf_mats"]))
    cfg = H.xylo_oracle_cfg(g, demo.net)
    fs, G = float(g["fs"]), len(g["doa_list"])
    # sources at chosen grid directions, among them ones beyond 3G/4 (the reference's trimmed window raises there)
    t = np.arange(T_TOTAL) / fs
    f_lo, f_hi = g["bands"][0]
    src = np.sin(2 * np.pi * np.cumsum(f_lo + (f_hi - f_lo) * t / t[-1]) / fs)
    rng = np.random.default_rng(2)
    xs = []
    for k in (0.1, 0.4, 0.6, 0.85, 0.95):
        sig = signal_from_template(geo, (t, src, float(g["doa_list"][int(k * (G - 1))])))
        xs.append(sig + 0.3 * np.sqrt(np.mean(sig ** 2)) * rng.standard_normal(sig.shape))
    x = zero_tail(np.stack(xs).astype(np.float32), g)
    xsb = demo.stream_batch(5, MAX_FRAME)
    sp, ra, counts, calls = run_stream(xsb, x, peak_win=15)
    nan_cases = 0
    for s in range(5):
        ref_in = O.xylo_encode(cfg, x[s])[0]
        raster, _ = O.xylo_lif(cfg, ref_in)
        f0 = 0
        for c in calls:
            m = int(c["n_out"][s])
            if m == 0:
                assert c["doa"][s] == -1 and np.all(np.isnan(c["rate"][s])) and np.isnan(c["periodic_ml"][s])
                continue
            rows = raster[f0:f0 + m]
            f0 += m
            cnt = rows.sum(0, dtype=np.int32)
            assert np.array_equal(c["counts"][s], cnt)
            _, d0, d1 = O.xylo_rate_doa(cnt, G, 1, m, fs, 15)
            assert c["doa"][s] == d0 and c["doa_peak"][s] == d1
            rate = demo.extract_rate(rows)
            np.testing.assert_allclose(c["rate"][s], rate, rtol=1e-12, atol=0)
            assert abs(c["periodic_ml"][s] - demo.estimate_doa_from_rate(rate, "periodic_ml")) <= 1e-12
            try:
                tr = demo.estimate_doa_from_rate(rate, "trimmed_periodic_ml")
            except IndexError:
                tr = None
            if tr is None:
                nan_cases += 1
                assert np.isnan(c["trimmed_periodic_ml"][s]) and int(c["flags"][s]) & 2
            else:
                assert abs(c["trimmed_periodic_ml"][s] - tr) <= 1e-12 and not int(c["flags"][s]) & 2
        assert f0 == T_TOTAL
    assert nan_cases > 0


def _stress_net(g, rng, scale=None):
    net = H.xylo_network(g)
    n = net.w_in.shape[1]
    if scale is None:      # test_multi_spike_steps_saturation_and_bias's network
        net.threshold = rng.integers(1, 40, size=n).astype(np.int16)
        net.dash_syn = rng.integers(0, 6, size=n).astype(np.int8)
        net.dash_mem = rng.integers(0, 8, size=n).astype(np.int8)
        net.bias = rng.integers(-3, 4, size=n).astype(np.int16)
        net.weight_shift_in = 3
        net.max_spikes = 7
    else:                  # small weights: the host drops the int16 clamps (SAT_ISYN = SAT_V = false)
        net.w_in = np.clip(net.w_in.astype(np.int32) // scale, -127, 127).astype(np.int8)
        net.threshold = np.full(n, max(int(net.threshold[0]) // scale, 2), dtype=np.int16)
    return net


@pytest.mark.gpu
@pytest.mark.parametrize("name,scale", [("xylo_c3_bipolar", None), ("xylo_c3_bipolar", 8),
                                        ("xylo_3band_o2", None), ("xylo_3band_o2", 8)])
def test_network_state_across_push_boundaries(name, scale):
    """Multi-spike steps, the spike cap, bias, weight shift and saturation (and small-weight networks without clamps) on
    the tensor-core LIF (one band) and the event-loop LIF (three bands), with frame edges inside 8-step groups and
    24-step tiles."""
    g = H.load(name)
    net = _stress_net(g, np.random.default_rng(11), scale)
    eng = H.xylo_engine(g, net)
    cfg = H.xylo_oracle_cfg(g, net)
    x = zero_tail(H.xylo_synth_clips(g, 5, T_TOTAL, seed=5, int16=True), g)
    frames = (3, 29, 77, 101, 250, 13, 997, 530, 1000, 1000)
    assert sum(frames) == T_TOTAL
    got = run_stream(stream_batch(eng, 5), x, frames)
    check_against_clip(eng, x, got)
    for s in range(5):
        raster, counts = O.xylo_lif(cfg, got[0][s])
        assert np.array_equal(got[1][s], raster) and np.array_equal(got[2][s], counts)
    if scale is None:
        assert max(int(r.max()) for r in got[1]) == 7


@pytest.mark.gpu
def test_slots_are_independent():
    g = H.load("xylo_c3_bipolar")
    eng = H.xylo_engine(g)
    x = zero_tail(H.xylo_synth_clips(g, 7, 3000, seed=21), g)
    frames = (500, 700, 300, 1000, 500)
    # S = 1 equals the same slot inside S = 7
    sp7, ra7, c7, _ = run_stream(stream_batch(eng, 7), x, frames)
    sp1, ra1, c1, _ = run_stream(stream_batch(eng, 1), x[3:4], frames)
    assert np.array_equal(sp1[0], sp7[3]) and np.array_equal(ra1[0], ra7[3]) and np.array_equal(c1[0], c7[3])
    # reset slot 2 after two pushes: from there on it equals a fresh batch fed from that point, the others are unchanged
    xsb = stream_batch(eng, 7)
    fresh = stream_batch(eng, 7)
    t, rows = 0, [[] for _ in range(7)]
    frows = []
    for i, n in enumerate(frames):
        if i == 2:
            xsb.reset([2])
            rows[2] = []
        out = xsb.push(dev(x[:, t:t + n]), want_spikes_in=True)
        if i >= 2:
            fo = fresh.push(dev(x[:, t:t + n]), want_spikes_in=True)
            frows.append(fo["spikes_in"][2, :fo["n_out"][2]].cpu())
            assert out["n_out"][2] == fo["n_out"][2]
        for s in range(7):
            rows[s].append(out["spikes_in"][s, :out["n_out"][s]].cpu())
        t += n
    out = xsb.flush(want_spikes_in=True)
    fo = fresh.flush(want_spikes_in=True)
    for s in range(7):
        rows[s].append(out["spikes_in"][s, :out["n_out"][s]].cpu())
    frows.append(fo["spikes_in"][2, :fo["n_out"][2]].cpu())
    assert torch.equal(torch.cat(rows[2]), torch.cat(frows))
    for s in (0, 1, 3, 4, 5, 6):
        assert np.array_equal(torch.cat(rows[s]).numpy(), sp7[s]), s
    # a flushed slot returns n_out = 0 and leaves its rows unwritten until it is reset
    xsb = stream_batch(eng, 7)
    xsb.push(dev(x[:, :1000]))
    fl = xsb.flush([4])
    assert fl["n_out"][4] == xsb.latency and fl["n_out"].sum() == xsb.latency      # the rest of its 1000 samples
    sent = torch.full((7, 1000 + xsb.latency, eng.N_in), 9, dtype=torch.int8, device="cuda")
    n_out = np.zeros(7, dtype=np.int64)
    fr = dev(x[:, 1000:2000])
    N.check(N.lib().micloc_xylo_streams_push(xsb._h, C.c_void_p(fr.data_ptr()), N.F32, 1000, 7,
                                             C.c_void_p(sent.data_ptr()), None, None, None, None, 0, None,
                                             n_out.ctypes.data_as(C.c_void_p), eng._stream()))
    assert n_out[4] == 0 and np.all(np.delete(n_out, 4) == 1000)
    assert bool((sent[4] == 9).all()) and bool((sent[3, :1000] != 9).all())
    xsb.reset([4])
    assert xsb.push(dev(x[:, :1000]))["n_out"][4] == 1000 - xsb.latency


@pytest.mark.gpu
def test_flag_invariant_with_long_digital_silence():
    """Long exact-zero stretches (flat tops the latency does not cover) next to normal clips: the silent slots are
    flagged, the others stay bit-exact with bit 0 clear, and every slot with bit 0 clear is bit-exact."""
    g = H.load("xylo_c3_bipolar")
    net = H.xylo_network(g)
    eng = H.xylo_engine(g, net)
    x = zero_tail(H.xylo_synth_clips(g, 4, 48_000, seed=12, int16=True), g)
    x[1, 1500:44_000] = 0
    x[3, 20_000:30_000] = 0
    frames = (4800,) * 10
    xsb = stream_batch(eng, 4, 4800)
    sp, ra, counts, calls = run_stream(xsb, x, frames)
    flags_push = np.bitwise_or.reduce(np.stack([c["flags"] for c in calls[:-1]]), axis=0)
    flags_flush = calls[-1]["flags"]
    ref = O.xylo_run_batch(H.xylo_oracle_cfg(g, net), x, float(g["fs"]), win=0, nthreads=4, want_spikes=True)
    assert flags_push[1] & 1 and flags_flush[1] & 1
    assert not flags_push[0] & 1 and not flags_flush[0] & 1 and not flags_flush[2] & 1
    for s in range(4):
        if not flags_flush[s] & 1:
            assert np.array_equal(signed(sp[s], eng.CT, True), ref["spikes_signed"][s]), s
            assert np.array_equal(counts[s], ref["counts"][s]), s


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 300])
def test_launches_per_push_are_constant(S):
    g = H.load("xylo_c3_bipolar")
    eng = H.xylo_engine(g)
    xsb = stream_batch(eng, S, 600)
    lib = N.lib()
    fr = dev(np.zeros((S, 500, 7), dtype=np.int16))
    xsb.push(fr)
    n0 = lib.micloc_launch_count()
    xsb.push(fr)                                        # assembly, STHT, chain, LIF, DoA
    n1 = lib.micloc_launch_count()
    xsb.push(fr, want_spikes_in=True, want_raster=True)  # + the pos / neg split
    n2 = lib.micloc_launch_count()
    assert (n1 - n0, n2 - n1) == (5, 6)


def _raw_ctx(g, M, n_ba):
    """A micloc_xylo context through the C-ABI with a chosen microphone count / band-filter length (unipolar, zero
    weights)."""
    lib = N.lib()
    G = len(g["doa_list"])
    keep = dict(kernel=np.ascontiguousarray(g["kernel"], dtype=np.float64),
                sos=np.ascontiguousarray([[1.0, 0, 0, 1, 0, 0]]), b=np.ascontiguousarray(g["ba_b"][:1]),
                a=np.ascontiguousarray(g["ba_a"][:1]), w=np.zeros((2 * M, G), dtype=np.int8),
                thr=np.ones(G, dtype=np.int16), ds=np.ones(G, dtype=np.int8), dm=np.ones(G, dtype=np.int8))
    cfg = N.XyloConfig()
    cfg.num_mic, cfg.kernel_len, cfg.stht_kernel = M, len(keep["kernel"]), keep["kernel"].ctypes.data_as(N._dp)
    cfg.num_bands, cfg.n_sections, cfg.sos = 1, 1, keep["sos"].ctypes.data_as(N._dp)
    cfg.n_ba = n_ba
    cfg.ba_b = keep["b"].ctypes.data_as(N._dp) if n_ba else None
    cfg.ba_a = keep["a"].ctypes.data_as(N._dp) if n_ba else None
    cfg.robust_width, cfg.bipolar, cfg.num_hidden, cfg.num_doa = 12, 0, G, G
    cfg.w_in = keep["w"].ctypes.data_as(C.POINTER(C.c_int8))
    cfg.threshold = keep["thr"].ctypes.data_as(C.POINTER(C.c_int16))
    cfg.dash_syn = keep["ds"].ctypes.data_as(C.POINTER(C.c_int8))
    cfg.dash_mem = keep["dm"].ctypes.data_as(C.POINTER(C.c_int8))
    cfg.max_spikes = 31
    h = C.c_void_p()
    N.check(lib.micloc_xylo_create(C.byref(cfg), 0, C.byref(h)))
    return h


@pytest.mark.gpu
def test_errors():
    g = H.load("xylo_c3_bipolar")
    eng = H.xylo_engine(g)
    xsb = stream_batch(eng, 3, 100)
    with pytest.raises(ValueError):
        xsb.push(torch.zeros((3, 50, 7), dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        xsb.push(torch.zeros((3, 0, 7), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        xsb.push(torch.zeros((3, 101, 7), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        xsb.push(torch.zeros((3, 50, 6), dtype=torch.float32, device="cuda"))
    with pytest.raises(ValueError):
        xsb.reset([3])
    with pytest.raises(ValueError):
        xsb.flush([-1])
    with pytest.raises(ValueError):
        xsb.push(torch.zeros((3, 50, 7), dtype=torch.float32, device="cuda"), peak_win=4)
    lib = N.lib()
    from haghighatshoarmuir2024_b200.xylo_snn_localization import XyloStreamBatch

    class _Ctx:                       # what XyloStreamBatch needs of an engine
        def __init__(self, h):
            self._h, self.device = h, torch.device("cuda", 0)
            self.M = self.F = self.G = self.N = self.N_in = 1

    for M, n_ba, code in ((7, 0, N.ERR_CONFIG), (33, 3, N.ERR_UNSUPPORTED)):
        h = _raw_ctx(g, M, n_ba)
        try:
            with pytest.raises(N.MiclocError) as e:
                XyloStreamBatch(_Ctx(h), 4, 100)
            assert e.value.code == code
        finally:
            lib.micloc_xylo_destroy(h)


def test_create_with_null_context_is_rejected_before_touching_the_gpu():
    lib = N.lib()
    h = C.c_void_p()
    assert lib.micloc_xylo_streams_create(None, 4, 100, C.byref(h)) == N.ERR_CONFIG
    assert b"null" in lib.micloc_last_error() and not h.value
