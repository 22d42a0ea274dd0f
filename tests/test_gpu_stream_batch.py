"""Stream batches (micloc_snn_streams_*, engine.SnnStreamBatch): many live recordings advanced by one push.

Every slot must give what the one-shot staged path gives on its own recording (a clip whose last K/2 samples are zero,
so that the stream's causal in-phase delay coincides with np.roll), bit for bit, and through it the float64 oracle."""
import numpy as np
import pytest
import torch

import helpers as H
from oracle import oracle as O

pytestmark = pytest.mark.gpu

RAGGED = [1, 31, 32, 33, 700, 4096, 2, 609, 4096]          # frame edges inside and on 32-sample blocks


def make_engine(g, T):
    from haghighatshoarmuir2024_b200.engine import SnnEngine
    return SnnEngine(H.chain_spec(g, T), g["bf_mat"], device=0)


def clips(g, S, T, seed, snrs=(-5.0, 0.0, 10.0, 20.0, 30.0), int16=False):
    """S recordings with their own seed and SNR, last K/2 samples zero: [S, T, M]."""
    xs = [H.synth_clips(g, 1, T, seed=seed + 7 * s, snrs_db=(snrs[s % len(snrs)],), int16=int16)[0][0] for s in range(S)]
    x = np.stack(xs)
    x[:, T - len(g["kernel"]) // 2:] = 0
    return x


def to_frames(x, dtype, junk=True):
    """[S, T, M] numpy -> device frames of `dtype`; int32 gets the recorder's 8th channel of junk."""
    xd = torch.from_numpy(x).cuda()
    if dtype == torch.int32:
        xd = xd.to(torch.int32)
        if junk:
            xd = torch.cat([xd, torch.full(xd.shape[:2] + (1,), 12345, dtype=torch.int32, device="cuda")], dim=2)
    return xd


def run_batch(sb, xd, lens, want_env=False, keys=("spikes",)):
    """Push the frame list through every slot, flush; per slot the concatenated final rows of `keys` + per-call dicts."""
    S = sb.num_streams
    parts = {k: [[] for _ in range(S)] for k in keys}
    calls = []
    t = 0
    for n in lens:
        out = sb.push(xd[:, t:t + n], want_env=want_env)
        t += n
        calls.append(out)
    assert t == xd.shape[1]
    calls.append(sb.flush(want_env=want_env))
    for out in calls:
        for s in range(S):
            m = int(out["n_out"][s])
            for k in keys:
                if m:
                    parts[k][s].append(out[k][s, :m])
    cat = {k: [torch.cat(v) if v else None for v in parts[k]] for k in keys}
    return cat, calls


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16, torch.int32])
def test_each_slot_equals_its_own_clip_bit_for_bit(dtype):
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    T, S = sum(RAGGED), 5
    x = clips(g, S, T, seed=21, int16=dtype != torch.float32)
    eng = make_engine(g, T)
    one = eng.run_taps(torch.from_numpy(x).cuda(), want=("spikes",))
    sb = SnnStreamBatch(eng, S, max_frame_len=4096)
    cat, calls = run_batch(sb, to_frames(x, dtype), RAGGED)
    assert calls[-1]["flags"].tolist() == [0] * S
    n_tot = np.sum([c["n_out"] for c in calls], axis=0)
    assert n_tot.tolist() == [T] * S
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / float(g["fs"]), float(g["tau"]), float(g["tau"]))
    for s in range(S):
        assert torch.equal(cat["spikes"][s], one["spikes"][s]), s
        ref = O.snn_apply(cfg, x[s].astype(np.float64), want=("spikes",))
        assert H.spike_agreement(cat["spikes"][s].cpu().numpy(), ref["spikes"]) >= 0.999


def test_power_and_doa_per_push_match_the_membrane_window():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    T, S = 9600, 3
    x = clips(g, S, T, seed=5, snrs=(15.0, 0.0, 25.0))
    eng = make_engine(g, T)
    vm = eng.run_taps(torch.from_numpy(x).cuda(), want=("vmem",))["vmem"].cpu().numpy().astype(np.float64)
    sb = SnnStreamBatch(eng, S, max_frame_len=4800)
    _, calls = run_batch(sb, torch.from_numpy(x).cuda(), [1000, 3800, 4800])
    lo = np.zeros(S, dtype=np.int64)
    for out in calls:
        for s in range(S):
            n = int(out["n_out"][s])
            if not n:
                continue
            power = np.mean((vm[s, lo[s]:lo[s] + n] @ g["bf_mat"]) ** 2, axis=0)
            assert H.rel_err(out["power"][s].cpu().numpy(), power) <= 1e-4
            assert int(out["doa"][s]) == int(np.argmax(power))
            lo[s] += n
    assert lo.tolist() == [T] * S


def test_envelope_per_slot_equals_the_one_shot_envelope():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch, envelope
    g = H.load("snn_c1_bipolar")
    T, S = 6000, 3
    x = clips(g, S, T, seed=3, snrs=(20.0, 5.0, 10.0))
    eng = make_engine(g, T)
    y = eng.run_taps(torch.from_numpy(x).cuda(), want=("y",))["y"]
    sb = SnnStreamBatch(eng, S, max_frame_len=2048)
    cat, _ = run_batch(sb, torch.from_numpy(x).cuda(), [2048, 2048, T - 4096], want_env=True, keys=("env", "doa_t"))
    for s in range(S):
        env_ref, idx_ref = envelope(y[s], 48000.0, 10e-3, 100e-3, want_argmax=True)
        assert torch.equal(cat["env"][s], env_ref) and torch.equal(cat["doa_t"][s], idx_ref), s


def test_slots_are_independent_under_reset_and_flush():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    half = len(g["kernel"]) // 2
    lens = [1000, 1000, 3000, 3000]
    T, S = sum(lens), 5
    x = clips(g, S, T, seed=40)
    x[[0, 3], 2000 - half:2000] = 0                        # slots 0 and 3 end after two frames in run C
    x_new = clips(g, 1, T - 2000, seed=99)[0]              # slot 2's second recording in run B
    eng = make_engine(g, T)
    xd = torch.from_numpy(x).cuda()

    def push_all(sb, frames_of, after_push=None):
        calls, t = [], 0
        for i, n in enumerate(lens):
            calls.append(sb.push(frames_of(i, t, n)))
            t += n
            if after_push:
                after_push(i, calls)
        calls.append(sb.flush())
        return calls

    def rows(calls, s, first=0):
        parts = [c["spikes"][s, :int(c["n_out"][s])] for c in calls[first:] if c["n_out"][s]]
        return torch.cat(parts)

    sb = SnnStreamBatch(eng, S, max_frame_len=3000)
    base = push_all(sb, lambda i, t, n: xd[:, t:t + n])

    # run B: slot 2 is reset after the second push and fed a new recording
    def frames_b(i, t, n):
        f = xd[:, t:t + n].clone()
        if i >= 2:
            f[2] = torch.from_numpy(x_new[t - 2000:t - 2000 + n]).cuda()
        return f
    sb.reset()
    run_b = push_all(sb, frames_b, lambda i, calls: sb.reset([2]) if i == 1 else None)
    for s in (0, 1, 3, 4):
        for cb, ca in zip(run_b, base):
            assert cb["n_out"][s] == ca["n_out"][s]
            m = int(ca["n_out"][s])
            assert torch.equal(cb["spikes"][s, :m], ca["spikes"][s, :m])
            if m:
                assert torch.equal(cb["power"][s], ca["power"][s]) and int(cb["doa"][s]) == int(ca["doa"][s])
    one_new = eng.run_taps(torch.from_numpy(x_new).cuda(), want=("spikes",))["spikes"][0]
    assert torch.equal(rows(run_b, 2, first=2), one_new)

    # run C: slots 0 and 3 are flushed after the second push; they return their tails, then nothing
    sb.reset()
    tails = {}
    run_c = push_all(sb, lambda i, t, n: xd[:, t:t + n],
                     lambda i, calls: tails.setdefault("f", sb.flush([0, 3])) if i == 1 else None)
    f = tails["f"]
    assert [int(v) for v in f["n_out"]] == [sb.latency, 0, 0, sb.latency, 0]
    short = eng.run_taps(torch.from_numpy(np.ascontiguousarray(x[[0, 3], :2000])).cuda(), want=("spikes",))["spikes"]
    for k, s in enumerate((0, 3)):
        got = torch.cat([c["spikes"][s, :int(c["n_out"][s])] for c in run_c[:2] + [f] if c["n_out"][s]])
        assert torch.equal(got, short[k])
        assert all(int(c["n_out"][s]) == 0 for c in run_c[2:])
    for s in (1, 2, 4):
        assert torch.equal(rows(run_c, s), rows(base, s))


def test_overflow_flag_stays_in_its_slot():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    T, S = 19200, 3
    x = clips(g, S, T, seed=8, snrs=(10.0,))
    x[1, 2000:14000] = 0                                     # 250 ms of digital silence, then the signal resumes
    eng = make_engine(g, T)
    sb = SnnStreamBatch(eng, S, max_frame_len=4800)
    _, calls = run_batch(sb, torch.from_numpy(x).cuda(), [4800] * 4)
    assert [int(v) & 1 for v in calls[-1]["flags"]] == [0, 1, 0]


def test_wide_array_tensor_core_stht():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_linear16")
    T, S = 6000, 3
    x = clips(g, S, T, seed=12, snrs=(10.0, 20.0, 0.0))
    eng = make_engine(g, T)
    one = eng.run_taps(torch.from_numpy(x).cuda(), want=("spikes",))["spikes"].cpu().numpy()
    sb = SnnStreamBatch(eng, S, max_frame_len=2048)
    cat, _ = run_batch(sb, torch.from_numpy(x).cuda(), [2048, 1000, 33, 2048, T - 5129])
    cfg = H.oracle_cfg(g)
    cfg.nir = O.neuron_kernel(np.arange(T) / float(g["fs"]), float(g["tau"]), float(g["tau"]))
    for s in range(S):
        got = cat["spikes"][s].cpu().numpy()
        assert got.shape == (T, 32)
        assert H.spike_agreement(got, one[s]) >= 0.999
        ref = O.snn_apply(cfg, x[s].astype(np.float64), want=("spikes",))
        assert H.spike_agreement(got, ref["spikes"]) >= 0.999


def test_many_slots_short_frames():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    lens = [100, 37, 263, 300, 200]
    T, S = sum(lens), 1024
    x, _ = H.synth_clips(g, S, T, seed=77)
    x[:, T - len(g["kernel"]) // 2:] = 0
    eng = make_engine(g, T)
    one = eng.run_taps(torch.from_numpy(x).cuda(), want=("spikes",))["spikes"]
    sb = SnnStreamBatch(eng, S, max_frame_len=300)
    cat, calls = run_batch(sb, torch.from_numpy(x).cuda(), lens)
    assert (np.sum([c["n_out"] for c in calls], axis=0) == T).all()
    for s in np.random.default_rng(0).choice(S, 8, replace=False).tolist() + [S - 1]:
        assert torch.equal(cat["spikes"][s], one[s]), s


def test_launches_per_push_do_not_grow_with_slots():
    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    eng = make_engine(g, 4800)
    lib = N.lib()
    counts = {}
    for S in (1, 64):
        sb = SnnStreamBatch(eng, S, max_frame_len=480)
        x = torch.randn((S, 480, 7), device="cuda")
        for want_env in (False, True):
            sb.push(x, want_env=want_env)                   # first request: envelope scratch
            c0 = lib.micloc_launch_count()
            sb.push(x, want_env=want_env)
            counts[(S, want_env)] = lib.micloc_launch_count() - c0
        sb.close()
    assert counts == {(1, False): 5, (64, False): 5, (1, True): 8, (64, True): 8}


def test_batch_argument_errors():
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    g = H.load("snn_c1_bipolar")
    eng = make_engine(g, 4800)
    with pytest.raises(ValueError):
        SnnStreamBatch(eng, 0, max_frame_len=100)                                 # num_streams < 1
    S = 4
    sb = SnnStreamBatch(eng, S, max_frame_len=100)
    with pytest.raises(ValueError):
        sb.push(torch.zeros((S, 50, 6), device="cuda"))                           # fewer channels than microphones
    with pytest.raises(ValueError):
        sb.push(torch.zeros((S, 101, 7), device="cuda"))                          # longer than max_frame_len
    with pytest.raises(ValueError):
        sb.push(torch.zeros((S, 0, 7), device="cuda"))                            # empty frame
    with pytest.raises(ValueError):
        sb.push(torch.zeros((S, 50, 7), dtype=torch.float64, device="cuda"))      # dtype
    with pytest.raises(ValueError):
        sb.push(torch.zeros((S + 1, 50, 7), device="cuda"))                       # slot count
    with pytest.raises(ValueError):
        sb.reset([S])                                                             # slot index out of range
    with pytest.raises(ValueError):
        sb.flush([-1])
    sb.push(torch.zeros((S, 100, 7), device="cuda"))
    out = sb.flush()
    assert out["n_out"].tolist() == [100] * S
    out = sb.push(torch.zeros((S, 100, 7), device="cuda"))                        # every slot flushed: nothing, no error
    assert out["n_out"].tolist() == [0] * S
    sb.reset([1])
    out = sb.push(torch.zeros((S, 100, 7), device="cuda"))
    assert out["n_out"].tolist() == [0] * S                                       # shorter than the latency
    assert sb.flush([1])["n_out"].tolist() == [0, 100, 0, 0]
