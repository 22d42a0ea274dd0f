"""Hilbert stream batches (micloc_hilbert_streams_*, beamformer.HilbertStreamBatch / Beamformer.stream_batch): the
Hilbert beamformer over many live recordings, band-pass, STHT history and filterbank state carried across pushes.
Needs a B200: run with -m gpu.

The analytic signal z of a slot's concatenated pushes must equal the one-shot chain's z of the whole recording bit
for bit (run_taps' z tap; with a filterbank, micloc_filterbank of the whole recording followed by a one-band batch).
On the 64-microphone array the STHT runs on the tensor cores, which scale each tile by its own largest magnitude, so
there the bit-for-bit comparison runs with MICLOC_STHT_FP32 set and the tensor-core z is held to 4e-5 of max |z|.
cov and power of every push are checked against a float64 restatement from the push's own z tap with the bounds of
test_gpu_hilbert_localize.py; the fused outputs against micloc_power_fuse on the push's own per-band power, bit for
bit."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
import test_gpu_hilbert_localize as HL
import test_gpu_power_paths as PP

pytestmark = pytest.mark.gpu

RAGGED = [1, 31, 32, 33, 700, 4096, 2, 609, 4096]          # frame edges inside and on 32-sample blocks
BANDS = [[1000.0, 1400.0], [1600.0, 2000.0], [2200.0, 2600.0]]
TC_Z_REL = 4e-5                 # tensor-core STHT tiles (5.3e-6 measured on one B200 at 1000 W)
ptr = lambda t: None if t is None else C.c_void_p(t.data_ptr())


def lib():
    from haghighatshoarmuir2024_b200 import _native as N
    return N, N.lib()


def sos_bank(F=3):
    from haghighatshoarmuir2024_b200.filterbank import ButterworthFilterbank
    return ButterworthFilterbank(BANDS[:F], order=2, fs=48_000.0)


class Batch:
    """micloc_hilbert_streams_* over SnnEngine contexts (their Hilbert steering matrices set)."""

    def __init__(self, engines, S, max_frame, bank=None, doa_list=None):
        N, L = lib()
        self.N, self.L, self.S, self.F = N, L, S, len(engines)
        self.M, self.G = engines[0].M, engines[0].hilbert_G
        self.sos = None if bank is None else np.ascontiguousarray(bank.sos_list, dtype=np.float64)
        self.doa = None if doa_list is None else np.ascontiguousarray(doa_list, dtype=np.float64)
        self.h = C.c_void_p()
        N.check(create(engines, S, max_frame, self.sos, self.doa, out=self.h))

    def push(self, frames, want=("z",), n_out=None):
        S, n, ch = frames.shape
        F, M, G, d = self.F, self.M, self.G, "cuda"
        mk = lambda k, shape, dt: torch.full(shape, -7, dtype=dt, device=d) if k in want else None
        o = {"z": mk("z", (F, S, n, 2 * M), torch.float32), "cov": mk("cov", (F, S, M, M, 2), torch.float64),
             "power": mk("power", (F, S, G), torch.float32), "power_grid": mk("power_grid", (S, G), torch.float32),
             "doa": mk("doa", (S,), torch.int32), "ml": mk("ml", (S,), torch.float64),
             "trimmed": mk("trimmed", (S,), torch.float64), "sumsq": mk("sumsq", (S,), torch.float64),
             "flags": mk("flags", (S,), torch.int32)}
        code = {torch.float32: self.N.F32, torch.int16: self.N.I16, torch.int32: self.N.I32}[frames.dtype]
        n_out = np.zeros(S, dtype=np.int64) if n_out is None else n_out
        self.N.check(self.L.micloc_hilbert_streams_push(
            self.h, ptr(frames), code, n, ch, ptr(o["z"]), ptr(o["cov"]), ptr(o["power"]), ptr(o["power_grid"]),
            ptr(o["doa"]), ptr(o["ml"]), ptr(o["trimmed"]), ptr(o["sumsq"]), ptr(o["flags"]),
            n_out.ctypes.data_as(C.c_void_p), None))
        assert n_out.tolist() == [n] * S
        return {k: v for k, v in o.items() if v is not None}

    def reset(self, slots=None):
        arr = None if slots is None else np.ascontiguousarray(slots, dtype=np.int32)
        self.N.check(self.L.micloc_hilbert_streams_reset(self.h, None if arr is None else arr.ctypes.data_as(C.c_void_p),
                                                         0 if arr is None else len(arr), None))

    def close(self):
        if self.h:
            self.L.micloc_hilbert_streams_destroy(self.h)
            self.h = None


def create(engines, S, max_frame, sos=None, doa=None, F=None, out=None):
    N, L = lib()
    ctxs = (C.c_void_p * max(len(engines), 1))(*[e._h.value for e in engines])
    h = C.c_void_p() if out is None else out
    rc = L.micloc_hilbert_streams_create(ctxs, len(engines) if F is None else F, 0 if sos is None else sos.shape[1],
                                         None if sos is None else sos.ctypes.data_as(N._dp),
                                         None if doa is None else doa.ctypes.data_as(N._dp), S, max_frame, C.byref(h))
    if out is None and rc == 0:
        L.micloc_hilbert_streams_destroy(h)
    return rc


def recordings(g, S, T, seed, dtype):
    """S recordings [S, T, M] whose last K/2 samples are zero (the stream's causal delay then equals np.roll), as
    (device frames of `dtype` with one junk channel, the same recording as float32 / int16 device clips for the
    one-shot paths)."""
    x = PP.clips(g, S, T, seed=seed, int16=dtype != torch.float32)
    x[:, T - len(g["kernel"]) // 2:] = 0
    if dtype == torch.int32:
        lo = np.random.default_rng(seed).integers(0, 1 << 16, x.shape)
        x = x.astype(np.int32) * 65536 + np.where(x != 0, lo, 0).astype(np.int32)
    one = torch.from_numpy(x).cuda()
    if dtype == torch.int32:
        one = one.to(torch.float32)                        # the stream's int32 -> float32 conversion (round to nearest)
    junk = np.full(x.shape[:2] + (1,), 1234, dtype=x.dtype)
    return torch.from_numpy(np.concatenate([x, junk], axis=2)).cuda(), one


def run(batch, frames, lens, want=("z",)):
    calls, t = [], 0
    for n in lens:
        calls.append(batch.push(frames[:, t:t + n].contiguous(), want=want))
        t += n
    assert t == frames.shape[1]
    return calls


def filterbank_rows(bank, frames, M):
    """micloc_filterbank of frames [S, T, ch] -> (rows [F, S, T, M], sumsq [S])."""
    N, L = lib()
    code = {torch.float32: N.F32, torch.int16: N.I16, torch.int32: N.I32}[frames.dtype]
    sos = np.ascontiguousarray(bank.sos_list, dtype=np.float64)
    S, T, ch = frames.shape
    out = torch.empty((sos.shape[0], S, T, M), dtype=torch.float32, device="cuda")
    ss = torch.empty(S, dtype=torch.float64, device="cuda")
    N.check(L.micloc_filterbank(ptr(frames), code, S, T, ch, M, sos.shape[0], sos.shape[1], sos.ctypes.data_as(N._dp),
                                ptr(out), ptr(ss), 0, None))
    return out, ss


def launches(want, F, wide):
    """The header's count: assembly, per band STHT + Gram kernel(s) (+ finish), + fuse."""
    finish = any(k in want for k in ("cov", "power", "power_grid", "doa", "ml", "trimmed", "flags"))
    fuse = any(k in want for k in ("power_grid", "doa", "ml", "trimmed", "flags"))
    return 1 + F * (2 + int(wide) + int(finish)) + int(fuse)


# ---------------------------------------------------------------------------
# 1. concatenation rule
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.int16, torch.int32])
@pytest.mark.parametrize("M", [7, 64])
def test_concatenated_z_equals_one_shot(M, dtype, monkeypatch):
    T, S = sum(RAGGED), 3
    g, eng, W = HL.hilbert_engine(M, 37, seed=M)
    frames, one = recordings(g, S, T, seed=M + 1, dtype=dtype)
    if M > 8:
        hb = Batch([eng], S, 4096)
        z_tc = torch.cat([c["z"][0] for c in run(hb, frames, RAGGED)], dim=1)
        ref_tc = eng.run_taps(one, want=("z",))["z"]
        e = PP.rel_err(z_tc.cpu().numpy(), ref_tc.cpu().numpy())
        PP.report(f"hilbert stream tensor-core z M={M} {dtype}", rel=e)
        assert e < TC_Z_REL
        hb.close()
        monkeypatch.setenv("MICLOC_STHT_FP32", "1")
    hb = Batch([eng], S, 4096)
    z = torch.cat([c["z"][0] for c in run(hb, frames, RAGGED)], dim=1)
    ref = eng.run_taps(one, want=("z",))["z"]
    for s in range(S):
        assert torch.equal(z[s], ref[s]), s


@pytest.mark.parametrize("dtype", [torch.float32, torch.int16, torch.int32])
def test_filterbank_bands_equal_one_band_batches_on_the_filterbank_output(dtype):
    T, S, M, bank = sum(RAGGED), 3, 7, sos_bank()
    engs = [HL.hilbert_engine(M, 37, seed=f)[1] for f in range(3)]
    g = PP.array_case(M, 4)
    frames, _ = recordings(g, S, T, seed=4, dtype=dtype)
    hb = Batch(engs, S, 4096, bank=bank)
    z = torch.cat([c["z"] for c in run(hb, frames, RAGGED)], dim=2)          # [F, S, T, 2M]
    rows, _ = filterbank_rows(bank, frames, M)
    for f in range(3):
        one = Batch([engs[f]], S, 4096)
        zf = torch.cat([c["z"][0] for c in run(one, rows[f], RAGGED)], dim=1)
        assert torch.equal(z[f], zf), f
        one.close()


# ---------------------------------------------------------------------------
# 2. per-push cov and power
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("M", [7, 64])
def test_cov_and_power_per_push_and_summed(M, monkeypatch):
    monkeypatch.setenv("MICLOC_STHT_FP32", "1")
    T, S = sum(RAGGED), 2
    g, eng, W = HL.hilbert_engine(M, 37, seed=M + 5)
    frames, one = recordings(g, S, T, seed=9, dtype=torch.float32)
    hb = Batch([eng], S, 4096)
    tol = HL.GRAM64 if M <= 8 else HL.TILED_REL
    calls = run(hb, frames, RAGGED, want=("z", "cov", "power"))
    worst_c = worst_p = 0.0
    for c in calls:
        cov64, p64 = HL.restate(c["z"][0].cpu().numpy(), W, 0)
        ec = HL.cov_err(torch.view_as_complex(c["cov"][0]), cov64)
        p = c["power"][0].cpu().numpy()
        ep = PP.f64_excess(p, p64) if M <= 8 else PP.rel_err(p, p64)
        worst_c, worst_p = max(worst_c, ec), max(worst_p, ep)
        assert ec < tol and ep < tol, (ec, ep)
    total = sum(torch.view_as_complex(c["cov"][0]) for c in calls).cpu().numpy()
    ref = eng.hilbert(one, t_start=0, bandpass=True, want=("cov",))["cov"].cpu().numpy()
    es = PP.rel_err(np.stack([total.real, total.imag], -1), np.stack([ref.real, ref.imag], -1))
    PP.report(f"hilbert stream M={M}", cov=worst_c, power=worst_p, summed_cov=es)
    assert es < tol


# ---------------------------------------------------------------------------
# 3. fusion, sumsq and the Python batch
# ---------------------------------------------------------------------------
def test_fused_outputs_equal_power_fuse_and_sumsq_the_filterbank_sumsq():
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer, HilbertStreamBatch
    N, L = lib()
    c2 = H.load("bench_c2_bf")
    doa_list = np.asarray(c2["doa_list"], np.float64)
    G = len(doa_list)
    bank = sos_bank()
    geo = CenterCircularArray(4.5e-2, 7)
    bands = []
    for f, band in enumerate(BANDS):
        bf = Beamformer(geo, 10e-3, band)
        bf.verbose = False
        bands.append((bf, HL.steering(7, G, f)))
    S = 5
    hb = HilbertStreamBatch(bands, S, 4096, filterbank=bank, doa_list=doa_list)
    assert hb.latency == 0
    g = PP.array_case(7, 4)
    frames, _ = recordings(g, S, sum(RAGGED), seed=2, dtype=torch.int32)
    want = ("power", "power_grid", "doa", "periodic_ml", "trimmed_periodic_ml", "flags")
    seen_bad = False
    t = 0
    for n in RAGGED:
        fr = frames[:, t:t + n].contiguous()
        t += n
        o = hb.push(fr, want=want)
        assert o["n_out"].tolist() == [n] * S
        grid = torch.empty((S, G), device="cuda")
        doa = torch.empty(S, dtype=torch.int32, device="cuda")
        ml = torch.empty(S, dtype=torch.float64, device="cuda")
        tr = torch.empty(S, dtype=torch.float64, device="cuda")
        fl = torch.empty(S, dtype=torch.int32, device="cuda")
        dl = torch.from_numpy(doa_list).cuda()
        N.check(L.micloc_power_fuse(ptr(o["power"]), 3, S, G, ptr(dl), ptr(grid), ptr(doa), ptr(ml), ptr(tr), ptr(fl),
                                    0, None))
        assert torch.equal(o["power_grid"], grid) and torch.equal(o["doa"], doa) and torch.equal(o["flags"], fl)
        assert torch.equal(o["periodic_ml"], ml)
        assert torch.allclose(o["trimmed_periodic_ml"], tr, rtol=0, atol=0, equal_nan=True)
        seen_bad |= bool((fl & 2).any())
        _, ss = filterbank_rows(bank, fr, 7)
        np.testing.assert_allclose(o["sumsq"].cpu().numpy(), ss.cpu().numpy(), rtol=1e-12)
        rms = np.sqrt(ss.cpu().numpy() / (n * 7))
        assert o["active"].cpu().numpy().tolist() == (rms >= 1e-4 * (2 ** 31 - 1)).tolist()
        deg = doa_list[o["doa"].cpu().numpy()] * 180 / np.pi
        deg[~o["active"].cpu().numpy()] = np.nan
        np.testing.assert_allclose(o["doa_deg"].cpu().numpy(), deg)
    PP.report("hilbert stream fusion", trimmed_index_error_seen=float(seen_bad))


def test_beamformer_stream_batch_is_the_beamformers_own_chain():
    """Beamformer.stream_batch: frames through the beamformer's band-pass chain; z equals hilbert_signal's chain
    (run_taps) on the whole recording, and the summed power over the pushes equals localize's power of it."""
    from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
    from haghighatshoarmuir2024_b200.beamformer import Beamformer
    gb = H.load("beamformer")
    bf = Beamformer(CenterCircularArray(4.5e-2, 7), 10e-3, list(gb["band"]), fs=float(gb["fs"]))
    bf.verbose = False
    x = np.asarray(gb["x"], np.float32).copy()
    K = len(bf.kernel)
    x[len(x) - K // 2:] = 0
    T = len(x)
    lens = [700, 33, T - 733]
    sb = bf.stream_batch(gb["bf_mat"], 1, max_frame_len=max(lens))
    xd = torch.from_numpy(x).cuda()
    outs, t = [], 0
    for n in lens:
        outs.append(sb.push(xd[None, t:t + n], want=("z", "power")))
        t += n
    z = torch.cat([o["z"][0, 0] for o in outs])
    assert torch.equal(z, bf._engine().run_taps(xd, want=("z",))["z"][0])
    p = sum(n * o["power"][0, 0].double() for n, o in zip(lens, outs)) / T
    ref = bf.localize(gb["bf_mat"], xd[None])["power"][0].double()
    assert PP.rel_err(p.cpu().numpy()[None], ref.cpu().numpy()[None]) < 1e-5
    sb.close()


# ---------------------------------------------------------------------------
# 4. slots
# ---------------------------------------------------------------------------
def test_slot_reset_and_single_slot():
    M, S = 7, 4
    lens = [1000, 1000, 3000, 3000]
    g, eng, W = HL.hilbert_engine(M, 37, seed=3)
    frames, _ = recordings(g, S, sum(lens), seed=40, dtype=torch.int16)
    new, _ = recordings(g, 1, sum(lens) - 2000, seed=99, dtype=torch.int16)
    want = ("z", "cov", "power")
    hb = Batch([eng], S, 3000)
    base = run(hb, frames, lens, want=want)
    hb.reset()
    run_b, t = [], 0
    for i, n in enumerate(lens):
        fr = frames[:, t:t + n].clone()
        if i >= 2:
            fr[2] = new[0, t - 2000:t - 2000 + n]
        run_b.append(hb.push(fr, want=want))
        t += n
        if i == 1:
            hb.reset([2])
    for ca, cb in zip(base, run_b):
        for s in (0, 1, 3):
            assert all(torch.equal(ca[k][:, s], cb[k][:, s]) for k in want), s
    fresh = Batch([eng], 1, 3000)
    one = run(fresh, new, lens[2:], want=want)
    for ca, cb in zip(one, run_b[2:]):
        assert all(torch.equal(ca[k][:, 0], cb[k][:, 2]) for k in want)
    single = Batch([eng], 1, 3000)
    for ca, cb in zip(run(single, frames[:1], lens, want=want), base):
        assert all(torch.equal(ca[k][:, 0], cb[k][:, 0]) for k in want)


# ---------------------------------------------------------------------------
# 5. contract
# ---------------------------------------------------------------------------
WANTS = [("z",), ("cov",), ("power",), ("doa",), ("flags",), ("z", "cov", "power", "power_grid", "doa", "ml", "trimmed")]


@pytest.mark.parametrize("case", ["narrow", "bank", "wide"])
def test_launches_per_push(case):
    N, L = lib()
    M = 64 if case == "wide" else 7
    F = 3 if case == "bank" else 1
    engs = [HL.hilbert_engine(M, 37, seed=f)[1] for f in range(F)]
    g = PP.array_case(M, 4)
    doa = np.linspace(-np.pi, np.pi, 37, endpoint=False)
    for want in WANTS:
        counts = {}
        for S in (1, 64):
            hb = Batch(engs, S, 480, bank=sos_bank() if F > 1 else None, doa_list=doa)
            x, _ = recordings(g, S, 480, seed=2, dtype=torch.int32)
            hb.push(x, want=want)
            c0 = L.micloc_launch_count()
            hb.push(x, want=want)
            counts[S] = L.micloc_launch_count() - c0
            hb.close()
        assert counts == {1: launches(want, F, M > 8), 64: launches(want, F, M > 8)}, (want, counts)


def test_push_does_not_synchronise():
    g, eng, W = HL.hilbert_engine(7, 37)
    hb = Batch([eng], 256, 4800)
    x, _ = recordings(g, 256, 4800, seed=1, dtype=torch.int32)
    hb.push(x, want=("cov", "power", "doa"))
    torch.cuda.synchronize()
    stream = torch.cuda.current_stream()
    torch.cuda._sleep(int(2e9))
    hb.push(x, want=("z", "cov", "power", "doa"))
    assert not stream.query()
    torch.cuda.synchronize()


def test_argument_errors():
    N, L = lib()
    M, S = 7, 4
    engs = [HL.hilbert_engine(M, 37, seed=f)[1] for f in range(3)]
    sos = np.ascontiguousarray(sos_bank().sos_list, dtype=np.float64)
    g = PP.array_case(M, 4)
    bare = PP.engine(g, 4801)
    assert create([bare], S, 100) == N.ERR_CONFIG                             # no Hilbert steering matrix
    wide_g = HL.hilbert_engine(M, 38, seed=9)[1]
    assert create([engs[0], wide_g], S, 100, sos) == N.ERR_SHAPE              # G differs
    six = HL.hilbert_engine(6, 37, seed=9)[1]
    assert create([engs[0], six], S, 100, sos) == N.ERR_SHAPE                 # M differs
    assert create(engs, S, 100, sos, F=0) == N.ERR_CONFIG
    assert create(engs * 3, S, 100, sos, F=9) == N.ERR_CONFIG
    assert create(engs, S, 100) == N.ERR_CONFIG                               # sos == NULL with F > 1
    assert create(engs, S, 100, sos) == 0
    assert create([engs[0]], S, 100) == 0
    hb = Batch([engs[0]], S, 100)                                             # no filterbank, no doa_list
    x, _ = recordings(g, S, 101, seed=1, dtype=torch.int32)
    with pytest.raises(ValueError, match="filterbank"):
        hb.push(x[:, :50].contiguous(), want=("sumsq",))
    with pytest.raises(ValueError, match="doa_list"):
        hb.push(x[:, :50].contiguous(), want=("ml",))
    with pytest.raises(ValueError, match="doa_list"):
        hb.push(x[:, :50].contiguous(), want=("trimmed",))
    with pytest.raises(ValueError, match="1..100"):
        hb.push(x)                                                            # longer than max_frame_len
    with pytest.raises(ValueError, match="number of microphones"):
        hb.push(x[:, :50, :6].contiguous())                                   # fewer channels than microphones
    n_out = np.zeros(S, dtype=np.int64)
    fr = x[:, :50].contiguous()
    rc = L.micloc_hilbert_streams_push(hb.h, ptr(fr), 7, 50, 8, *([None] * 9), n_out.ctypes.data_as(C.c_void_p), None)
    assert rc == N.ERR_SHAPE and "dtype" in L.micloc_last_error().decode()
    assert hb.push(fr)["z"].shape == (1, S, 50, 2 * M)                        # the batch still works
    hb.close()
    bare.close()
