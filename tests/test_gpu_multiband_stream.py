"""Multi-band stream batches (micloc_snn_mb_streams_*, localization_demo_snn.MultibandStreamBatch): the live localiser
(filterbank -> one chain per band -> power summed over the bands -> estimators) with its state carried across pushes.

Every band must give, bit for bit, what micloc_filterbank of the whole recording followed by that band's
SnnStreamBatch gives; power and the estimators are checked against float64 numpy on the resulting spikes."""
import ctypes as C

import numpy as np
import pytest
import torch
from scipy.signal import lfilter

import helpers as H

pytestmark = pytest.mark.gpu

RAGGED = [1, 31, 32, 33, 700, 4096, 2, 609, 4096]          # frame edges inside and on 32-sample blocks
ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())


def make_demo(g, G449=False):
    """The full_multiband golden's localiser (G = 64), or config 2's steering matrices (G = 449) on the same bands."""
    from haghighatshoarmuir2024_b200.array_geometry import ArrayGeometry
    from haghighatshoarmuir2024_b200.localization_demo_snn import Demo
    if G449:
        c2 = H.load("bench_c2_bf")
        doa_list, bf_mats = c2["doa_list"], [c2[f"bf_{f}"] for f in range(3)]
    else:
        doa_list, bf_mats = g["doa_list"], list(g["bf_mats"])
    return Demo(geometry=ArrayGeometry(g["r_vec"], g["theta_vec"]), freq_bands=g["bands"], doa_list=doa_list,
                recording_duration=0.25, kernel_duration=float(g["kernel_duration"]), bipolar_spikes=bool(g["bipolar"]),
                fs=float(g["fs"]), bf_mats=bf_mats)


def recordings(g, S, T, seed, snrs=(30.0, 10.0, 0.0, 20.0)):
    """S recordings [S, T, 7] float64 in [-1, 1): the golden frame, shifted and scaled per slot, + white noise at the
    slot's SNR (own seed per slot)."""
    base = g["frame"][:, :7].astype(np.float64) / 2.0 ** 31
    base = np.resize(base.T, (7, T)).T
    out = []
    for s in range(S):
        rng = np.random.default_rng(seed + 11 * s)
        x = np.roll(base, int(rng.integers(0, T)), axis=0) * rng.uniform(0.5, 2.0)
        sig = np.sqrt(np.mean(x ** 2))
        out.append(x + rng.standard_normal(x.shape) * sig * 10 ** (-snrs[s % len(snrs)] / 20))
    return np.clip(np.stack(out), -0.99, 0.99)


def to_frames(x, dtype):
    """[S, T, 7] in [-1, 1) -> device frames of `dtype` with the recorder's 8th channel of junk."""
    scale = {torch.float32: 1.0, torch.int16: 2.0 ** 15, torch.int32: 2.0 ** 31}[dtype]
    npdt = {torch.float32: np.float32, torch.int16: np.int16, torch.int32: np.int32}[dtype]
    v = x * scale if dtype == torch.float32 else np.round(x * scale)
    junk = np.full(x.shape[:2] + (1,), 1234, dtype=np.float64)
    return torch.from_numpy(np.concatenate([v, junk], axis=2).astype(npdt)).cuda()


def filterbank(demo, frames):
    """micloc_filterbank of frames [S, T, ch] -> (rows [F, S, T, M] float32, sumsq [S] float64)."""
    from haghighatshoarmuir2024_b200 import _native as N
    code = {torch.float32: N.F32, torch.int16: N.I16, torch.int32: N.I32}[frames.dtype]
    sos = np.ascontiguousarray(demo.filterbank.sos_list, dtype=np.float64)
    S, T, ch = frames.shape
    F, M = sos.shape[0], demo.num_mic
    out = torch.empty((F, S, T, M), dtype=torch.float32, device="cuda")
    ss = torch.empty(S, dtype=torch.float64, device="cuda")
    N.check(N.lib().micloc_filterbank(ptr(frames), code, S, T, ch, M, F, sos.shape[1], sos.ctypes.data_as(N._dp),
                                      ptr(out), ptr(ss), 0, None))
    return out, ss


def run(mb, frames, lens, want_spikes=True):
    """Push the frame list through every slot, then flush: the list of per-call dicts."""
    calls, t = [], 0
    for n in lens:
        calls.append(mb.push(frames[:, t:t + n], want_spikes=want_spikes))
        t += n
    assert t == frames.shape[1]
    calls.append(mb.flush(want_spikes=want_spikes))
    return calls


def concat_spikes(calls, f, s):
    parts = [c["spikes"][f, s, :int(c["n_out"][s])] for c in calls if c["n_out"][s]]
    return torch.cat(parts)


def band_stream_spikes(demo, mb, frames, lens, slots):
    """Reference: micloc_filterbank of the whole recordings, band f's rows through an SnnStreamBatch on band f's engine
    with the same frame lengths: concatenated final spikes [F][len(slots)] of the listed slots."""
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    rows, _ = filterbank(demo, frames[slots])
    ref = []
    for f, eng in enumerate(mb.engines):
        sb = SnnStreamBatch(eng, len(slots), max_frame_len=mb.max_frame_len)
        parts = [[] for _ in slots]
        t = 0
        outs = []
        for n in lens:
            outs.append(sb.push(rows[f, :, t:t + n].contiguous()))
            t += n
        outs.append(sb.flush())
        assert outs[-1]["flags"].tolist() == [0] * len(slots)
        for o in outs:
            for k in range(len(slots)):
                if o["n_out"][k]:
                    parts[k].append(o["spikes"][k, :int(o["n_out"][k])])
        ref.append([torch.cat(p) for p in parts])
        sb.close()
    return ref


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16, torch.int32])
def test_bands_equal_single_band_streams_on_the_filterbank_output(dtype):
    g = H.load("full_multiband")
    demo = make_demo(g)
    T, S = sum(RAGGED), 4
    frames = to_frames(recordings(g, S, T, seed=3), dtype)
    mb = demo.stream_batch(S, max_frame_len=4096)
    calls = run(mb, frames, RAGGED)
    assert (np.sum([c["n_out"] for c in calls], axis=0) == T).all()
    assert [int(v) & 1 for v in calls[-1]["flags"]] == [0] * S          # bit 1: the trimmed estimator's IndexError
    ref = band_stream_spikes(demo, mb, frames, RAGGED, list(range(S)))
    for f in range(3):
        for s in range(S):
            assert torch.equal(concat_spikes(calls, f, s), ref[f][s]), (f, s)


def test_sumsq_per_push_is_the_filterbank_sumsq_of_the_frame():
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [700, 33, 4096, 1]
    S = 3
    frames = to_frames(recordings(g, S, sum(lens), seed=9), torch.int32)
    mb = demo.stream_batch(S, max_frame_len=4096)
    t = 0
    for n in lens:
        out = mb.push(frames[:, t:t + n])
        _, ss = filterbank(demo, frames[:, t:t + n].contiguous())
        np.testing.assert_allclose(out["sumsq"].cpu().numpy(), ss.cpu().numpy(), rtol=1e-12)
        t += n


def test_power_and_estimators_per_push_match_float64_numpy():
    """Per band, the membrane is recomputed in float64 from the pushed spikes (causal FIR with the engine's alpha
    taps).  Bound 5e-4 on power: the parity tests hold the float32 membrane to 1e-4 of float64, and power is quadratic
    in it (2 x 1e-4, plus the float32 membrane's rounding over the window), not a measured figure."""
    from haghighatshoarmuir2024_b200.engine import neuron_alpha_params
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [100, 2000, 4000, 3900]                      # the first push is shorter than the latency
    T, S = sum(lens), 3
    frames = to_frames(recordings(g, S, T, seed=5, snrs=(20.0, 5.0, 30.0)), torch.int32)
    mb = demo.stream_batch(S, max_frame_len=4000)
    calls = run(mb, frames, lens)
    G, doa_list = len(demo.doa_list), demo.doa_list
    ys = []                                             # [F][S] float64 beamformed membrane [T, G]
    for f in range(3):
        taps = neuron_alpha_params(mb.time_vec, demo.beamfs[f].tau_vec)[0]
        ys.append([lfilter(taps, [1.0], concat_spikes(calls, f, s).cpu().numpy().astype(np.float64), axis=0)
                   @ demo.bf_mats[f] for s in range(S)])
    lo = np.zeros(S, dtype=np.int64)
    for c in calls:
        for s in range(S):
            n = int(c["n_out"][s])
            if not n:
                continue
            dev_p = c["power"][:, s].cpu().numpy().astype(np.float64)
            for f in range(3):
                ref = np.mean(ys[f][s][lo[s]:lo[s] + n] ** 2, axis=0)
                assert H.rel_err(dev_p[f], ref) <= 5e-4, (f, s, lo[s])
            grid = dev_p.sum(0)                         # float64 sum in band order
            np.testing.assert_allclose(c["power_grid"][s].cpu().numpy(), grid, rtol=1e-6)
            idx = int(np.argmax(grid))
            assert int(c["doa"][s]) == idx
            assert abs(float(c["periodic_ml"][s]) - np.angle(np.mean(grid * np.exp(1j * doa_list)))) < 1e-9
            num = G // 2
            rng_idx = np.arange(-num // 2, num // 2 + 1) - idx
            fl = int(c["flags"][s])
            try:
                want = np.angle(np.mean(grid[rng_idx] * np.exp(1j * doa_list[rng_idx])))
                assert abs(float(c["trimmed_periodic_ml"][s]) - want) < 1e-9 and fl & 2 == 0
            except IndexError:
                assert np.isnan(float(c["trimmed_periodic_ml"][s])) and fl & 2 == 2
            lo[s] += n
    assert lo.tolist() == [T] * S


def test_one_latency_and_unwritten_rows():
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("full_multiband")
    demo = make_demo(g, G449=True)
    S, n_max = 2, 600
    mb = demo.stream_batch(S, max_frame_len=n_max)
    D = mb.latency
    lags = []
    for eng in mb.engines:
        sb = SnnStreamBatch(eng, 1, max_frame_len=16)
        lags.append(sb.latency)
        sb.close()
    assert lags == [8 * w + 33 for w in (12, 10, 9)] and D == max(lags) == 129
    F, G, C2 = 3, 449, 14
    frames = to_frames(recordings(g, S, 2000, seed=1), torch.int32)
    lib = N.lib()
    N_s = F_s = 0
    t = 0
    for n in (100, 28, 1, 600, 31, 600, 300):          # the first two pushes stay below D
        rows = n + D
        spikes = torch.full((F, S, rows, C2), 7, dtype=torch.int8, device="cuda")
        power = torch.full((F, S, G), -1.0, device="cuda")
        grid = torch.full((S, G), -1.0, device="cuda")
        doa = torch.full((S,), -5, dtype=torch.int32, device="cuda")
        ml = torch.full((S,), -9.0, dtype=torch.float64, device="cuda")
        tr = torch.full((S,), -9.0, dtype=torch.float64, device="cuda")
        fl = torch.full((S,), -3, dtype=torch.int32, device="cuda")
        ss = torch.empty(S, dtype=torch.float64, device="cuda")
        n_out = np.zeros(S, dtype=np.int64)
        fr = frames[:, t:t + n].contiguous()
        N.check(lib.micloc_snn_mb_streams_push(mb._h, ptr(fr), N.I32, n, 8, ptr(spikes), ptr(power), ptr(grid), ptr(doa),
                                               ptr(ml), ptr(tr), ptr(ss), ptr(fl), n_out.ctypes.data_as(C.c_void_p), None))
        torch.cuda.synchronize()
        t += n
        N_s += n
        want = max(N_s - D, F_s) - F_s
        assert n_out.tolist() == [want] * S
        F_s += want
        if want == 0:
            assert (spikes == 7).all() and (power == -1).all() and (grid == -1).all()
            assert (doa == -5).all() and (ml == -9).all() and (tr == -9).all() and (fl == -3).all()
        else:
            assert (spikes[:, :, :want] != 7).all() and (spikes[:, :, want:] == 7).all()
            assert (power >= 0).all() and (grid >= 0).all() and ((fl & ~2) == 0).all()


def test_golden_recording_streamed():
    """The full_multiband frame (12 000 x 8 int32) pushed in ragged frames.  The n_out-weighted mean of the per-push
    power_grid is the power of the whole recording, as the one-shot golden computes it, except for the in-phase branch
    of its first samples: the stream delays causally (zeros before the start), the golden rolls the clip (its last K/2
    = 240 samples).  That changes the band-passed in-phase input for t < 240, and the chain needs about
    7 fs / (pi BW) = 270 samples (BW = 400 Hz, decay to 1e-3) plus the neuron's ~40 taps to forget it: about 550 of the
    12 000 rows.  A row holds at most about twice the mean power of the steady tone, so the power grids differ by at
    most 2 x 550 / 12 000 ~ 0.09 of the peak (derived, not measured)."""
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = RAGGED + [2400]
    frame = torch.from_numpy(g["frame"]).cuda()[None]
    mb = demo.stream_batch(1, max_frame_len=4096)
    calls = run(mb, frame, lens, want_spikes=False)
    n = np.array([int(c["n_out"][0]) for c in calls])
    assert n.sum() == 12000 and int(calls[-1]["flags"][0]) & 1 == 0
    grid = sum(k * c["power_grid"][0].cpu().numpy().astype(np.float64) for k, c in zip(n, calls) if k) / n.sum()
    assert int(np.argmax(grid)) == int(g["doa"])
    assert H.rel_err(grid, g["power_grid"]) < 0.09


def test_slots_are_independent_under_reset_and_flush():
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [1000, 1000, 3000, 3000]
    T, S = sum(lens), 4
    frames = to_frames(recordings(g, S, T, seed=40), torch.int32)
    x_new = to_frames(recordings(g, 1, T - 2000, seed=99), torch.int32)[0]
    mb = demo.stream_batch(S, max_frame_len=3000)
    keys = ("spikes", "power", "power_grid", "doa", "periodic_ml", "trimmed_periodic_ml")

    def push_all(frames_of, after_push=None):
        calls, t = [], 0
        for i, n in enumerate(lens):
            calls.append(mb.push(frames_of(i, t, n), want_spikes=True))
            t += n
            if after_push:
                after_push(i)
        calls.append(mb.flush(want_spikes=True))
        return calls

    def same(ca, cb, s, key):
        m = int(ca["n_out"][s])
        if key == "spikes":
            return torch.equal(ca[key][:, s, :m], cb[key][:, s, :m])
        if not m:
            return True
        idx = (slice(None), s) if key == "power" else s
        return torch.equal(ca[key][idx], cb[key][idx]) or (      # bit for bit; NaN (IndexError case) == NaN
            ca[key].is_floating_point() and torch.allclose(ca[key][idx], cb[key][idx], rtol=0, atol=0, equal_nan=True))

    base = push_all(lambda i, t, n: frames[:, t:t + n])

    # run B: slot 2 is reset after the second push and fed a new recording
    def frames_b(i, t, n):
        f = frames[:, t:t + n].clone()
        if i >= 2:
            f[2] = x_new[t - 2000:t - 2000 + n]
        return f
    mb.reset()
    run_b = push_all(frames_b, lambda i: mb.reset([2]) if i == 1 else None)
    for s in (0, 1, 3):
        for ca, cb in zip(base, run_b):
            assert ca["n_out"][s] == cb["n_out"][s]
            assert all(same(ca, cb, s, k) for k in keys), s
    for ca, cb in zip(base[:-1], run_b[:-1]):
        assert torch.equal(ca["sumsq"][[0, 1, 3]], cb["sumsq"][[0, 1, 3]])
    fresh = demo.stream_batch(1, max_frame_len=3000)
    one = [fresh.push(x_new[None, :3000], want_spikes=True), fresh.push(x_new[None, 3000:], want_spikes=True),
           fresh.flush(want_spikes=True)]
    for ca, cb in zip(one, run_b[2:]):
        assert ca["n_out"][0] == cb["n_out"][2]
        m = int(ca["n_out"][0])
        assert torch.equal(ca["spikes"][:, 0, :m], cb["spikes"][:, 2, :m])
        if m:
            assert torch.equal(ca["power_grid"][0], cb["power_grid"][2]) and int(ca["doa"][0]) == int(cb["doa"][2])

    # run C: slots 0 and 3 are flushed after the second push; they return their tails, then nothing until reset
    mb.reset()
    tails = {}
    run_c = push_all(lambda i, t, n: frames[:, t:t + n],
                     lambda i: tails.setdefault("f", mb.flush([0, 3], want_spikes=True)) if i == 1 else None)
    assert tails["f"]["n_out"].tolist() == [mb.latency, 0, 0, mb.latency]
    for c in run_c[2:]:
        assert c["n_out"][0] == 0 and c["n_out"][3] == 0
    for s in (1, 2):
        for ca, cc in zip(base, run_c):
            assert ca["n_out"][s] == cc["n_out"][s]
            assert all(same(ca, cc, s, k) for k in keys), s
    mb.reset([0])
    assert mb.push(frames[:, :1000])["n_out"].tolist() == [1000 - mb.latency, 0, 0, 0]   # the others were flushed


def test_overflow_flag_stays_in_its_slot():
    """Half a second of digital silence, then signal, overflows the RZCC clusters of slot 1 (as it did when the batch
    was introduced).  The flush's host flags OR the bands' overflow bits: bit 0 for slot 1 only, as the fused flags of
    the last push report it."""
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [4800] * 10
    x = recordings(g, 3, sum(lens), seed=8)
    x[1, 4000:28000] = 0.0
    mb = demo.stream_batch(3, max_frame_len=4800)
    calls = run(mb, to_frames(x, torch.int32), lens, want_spikes=False)
    assert [int(v) & 1 for v in calls[-1]["flags"]] == [0, 1, 0]
    assert [int(v) & 1 for v in calls[-2]["flags"].cpu()] == [0, 1, 0]


def test_activity_gate():
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [2000, 2000, 2000]
    x = recordings(g, 3, sum(lens), seed=7)
    x[1] = 0.0
    frames = to_frames(x, torch.int32)
    mb = demo.stream_batch(3, max_frame_len=2000)
    t = 0
    for n in lens:
        out = mb.push(frames[:, t:t + n])
        t += n
        assert out["active"].cpu().tolist() == [True, False, True]
        deg = out["doa_deg"].cpu().numpy()
        assert np.isnan(deg[1]) and np.isfinite(deg[[0, 2]]).all()


def test_launches_per_push():
    from haghighatshoarmuir2024_b200 import _native as N
    g = H.load("full_multiband")
    demo = make_demo(g)
    lib = N.lib()
    counts = {}
    for S in (1, 64):
        mb = demo.stream_batch(S, max_frame_len=480)
        x = to_frames(recordings(g, S, 480, seed=2), torch.int32)
        mb.push(x)
        c0 = lib.micloc_launch_count()
        mb.push(x)
        counts[S] = lib.micloc_launch_count() - c0
        mb.close()
    assert counts == {1: 4 * 3 + 2, 64: 4 * 3 + 2}


def test_many_slots_short_frames():
    g = H.load("full_multiband")
    demo = make_demo(g)
    lens = [100, 37, 263, 300, 200]
    T, S = sum(lens), 1024
    rng = np.random.default_rng(77)
    x = recordings(g, 1, T, seed=77)[0][None] * rng.uniform(0.2, 1.0, (S, 1, 1))
    x = np.clip(x + rng.standard_normal(x.shape) * 0.01, -0.99, 0.99)
    frames = to_frames(x, torch.int32)
    mb = demo.stream_batch(S, max_frame_len=300)
    calls = run(mb, frames, lens)
    assert (np.sum([c["n_out"] for c in calls], axis=0) == T).all()
    slots = sorted(rng.choice(S, 6, replace=False).tolist() + [S - 1])
    ref = band_stream_spikes(demo, mb, frames, lens, slots)
    for f in range(3):
        for k, s in enumerate(slots):
            assert torch.equal(concat_spikes(calls, f, s), ref[f][k]), (f, s)


def test_argument_errors():
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.engine import SnnEngine
    g = H.load("full_multiband")
    demo = make_demo(g)
    lib = N.lib()
    S = 4
    mb = demo.stream_batch(S, max_frame_len=100)
    sos = np.ascontiguousarray(demo.filterbank.sos_list, dtype=np.float64)

    def create(engines, F=None):
        ctxs = (C.c_void_p * max(len(engines), 1))(*[e._h.value for e in engines])
        h = C.c_void_p()
        rc = lib.micloc_snn_mb_streams_create(ctxs, len(engines) if F is None else F, sos.shape[1],
                                              sos.ctypes.data_as(N._dp), None, S, 100, C.byref(h))
        if rc == 0:
            lib.micloc_snn_mb_streams_destroy(h)
        N.check(rc)

    spec = demo.beamfs[0].chain_spec(mb.time_vec)
    wide = SnnEngine(spec, np.random.default_rng(0).standard_normal((14, 65)))
    spec.num_mic = 6
    six = SnnEngine(spec, np.random.default_rng(0).standard_normal((12, 64)))
    with pytest.raises(ValueError, match="DoAs"):
        create([mb.engines[0], wide])                                         # G differs
    with pytest.raises(ValueError, match="microphones"):
        create([mb.engines[0], six])                                          # M differs
    with pytest.raises(ValueError, match="1..8"):
        create(mb.engines, F=0)
    with pytest.raises(ValueError, match="1..8"):
        create(mb.engines * 3, F=9)
    create(mb.engines)
    x = to_frames(recordings(g, S, 101, seed=1), torch.int32)
    with pytest.raises(ValueError, match="number of microphones"):
        mb.push(x[:, :50, :6])                                                # fewer channels than microphones
    with pytest.raises(ValueError, match="float32, int16 or int32"):
        mb.push(x[:, :50].to(torch.float64))
    with pytest.raises(ValueError, match="slots"):
        mb.push(x[:S - 1, :50])
    with pytest.raises(ValueError, match="number of microphones"):
        mb.push(x[:, :50, 0])                                                 # not [S, n, channels]
    with pytest.raises(ValueError, match="1..100"):
        mb.push(x)                                                            # longer than max_frame_len
    with pytest.raises(ValueError, match="out of range"):
        mb.reset([S])
    with pytest.raises(ValueError, match="out of range"):
        mb.flush([-1])
    assert mb.push(x[:, :100])["n_out"].tolist() == [0] * S                   # nothing was pushed before
