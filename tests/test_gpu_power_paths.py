"""Membrane, Gram, power and first-maximum DoA of every device path against a float64 restatement driven by the
kernels' own spikes.  Needs a B200: run with -m gpu.

Everything downstream of the spike decision is deterministic arithmetic, so it is checked exactly rather than through
the oracle (whose spikes differ from the device's in ~0.1 % of positions, which forces 2e-3 on power):

  membrane64   v[t] = sum_{n<L} c n a^n s[t-n] per channel, by its definition (scipy lfilter of the FIR)
  gram64       sum_{t >= t_start} v[t] v[t]^T in float64
  power64      diag(W^T G W) / T_rows with the float64 bf_mat W
  first_argmax the first index of the maximum
  cproject64   y = (z_re + i z_im) conj(bf) of the Hilbert beamformer

Power / DoA of the staged paths are compared with power64 of the call's own float32 `vmem` tap promoted to float64, so
that only the Gram / power arithmetic is under test.  Which Gram and power kernels a shape selects
(micloc_api.cu:run_power, micloc::launch_power):

  k_gram + k_power_argmax<true>    C2 = 2M < 32, or T < 256, or MICLOC_NO_SEGMENTS
  k_gram_slab + k_gram_reduce      C2 < 32, T >= 65536, B * ceil(C2^2 / 256) < 2 * SMs
  k_gram_tiled + k_gram_reduce     32 <= C2 < 64 (M = 16 ... 31), or MICLOC_GRAM_FP32
  k_gram_tc<true> + k_gram_reduce  64 <= C2 <= 128 (M = 32 ... 64)
  k_gram_tc<false>                 C2 > 128 (M = 65 ... 128): off-diagonal 128 x 128 blocks
  k_power_wide                     C2 >= 32 and C2^2 8 + (32 C2 + 256) 8 <= 200 KB (M <= 72)
  k_power_argmax<true>             C2 < 32, M = 73 ... 84, or MICLOC_POWER_NARROW (Gram in shared memory)
  k_power_argmax<false>            M >= 85: the Gram matrix no longer fits a block's shared memory, read from global
  DoA slices + k_argmax_chunks     B < SMs and G C2^2 >= 2^20

Tolerances.  `power` is stored as float32, so a float64 path is held to its excess over the float32 rounding of the
exact value (|p - p64| - 2^-24 |p64|, relative to the clip's largest power).  Every bound is below what dropping one
32-sample block would cause, 32 / (10 T) of the largest power, and about 10x the largest error measured on one B200
(1000 W power limit), in brackets:
  float64 Gram and power (k_gram, k_gram_slab, k_power_*, k_cpower_argmax, micloc_snn_gram)   0 excess    (1e-12)
  k_gram_tiled (float32 over 1024-sample slabs)                                          4.2e-7      (5e-6)
  k_gram_tc (fp16 hi/lo mma.sync, float32 over slabs; lo x lo dropped)                   5.6e-6      (6e-5)
  fused epilogues, against power64(membrane64(spikes))                                   9.5e-7      (1e-5)
  float32 membrane recursion against membrane64, of max |v|                              6.1e-7      (6e-6)
  k_dense / k_cproject float32 projections                                               3.3e-7      (4e-6)
"""
import ctypes as C
import time

import numpy as np
import pytest
import torch
from scipy.signal import lfilter

import helpers as H

pytestmark = pytest.mark.gpu

F64_EXCESS = 1e-12       # float64 products and sums, beyond the float32 rounding of the stored power
F32_REL = 5e-6           # k_gram_tiled: float32 products and sums over 1024-sample slabs
TC_REL = 6e-5            # k_gram_tc: fp16 hi/lo products on the tensor cores, float32 sums over slabs
FUSED_REL = 1e-5         # fused epilogues against power64(membrane64(spikes)): float32 membrane + tensor-core Gram
MEMBRANE_REL = 6e-6      # float32 neuron recursion against the float64 FIR, of max |v|
DENSE_REL = 4e-6         # k_dense / k_cproject float32 projections
U32 = 2.0 ** -24         # unit roundoff of float32


# ---------------------------------------------------------------------------
# float64 reference
# ---------------------------------------------------------------------------
def membrane64(spikes, a, c, L):
    """v[t] = sum_{n<L} c n a^n s[t-n] along the time axis (axis -2) of int8 spikes [..., T, C2]."""
    n = np.arange(L, dtype=np.float64)
    h = c * n * a ** n
    return lfilter(h, [1.0], np.asarray(spikes, np.float64), axis=-2)


def gram64(v, t_start=0):
    v = np.asarray(v, np.float64)[..., t_start:, :]
    return np.einsum("...tc,...td->...cd", v, v)


def power64(v, W, rows=None):
    """diag(W^T G W) / T_rows per clip of v [B, T, C2]."""
    v = np.asarray(v, np.float64)
    if rows is not None:
        return np.stack([power64(v[b:b + 1, :rows[b]], W)[0] for b in range(len(v))])
    G = gram64(v)
    return np.einsum("bcg,cg->bg", G @ W, W) / v.shape[1]


def first_argmax(p):
    return np.argmax(p, axis=-1)


def cproject64(z, bf_re, bf_im):
    """y[b,t,g] = sum_m (z_re + i z_im)[b,t,m] conj(bf[m,g]) for z [B, T, 2M] (real | imag)."""
    M = bf_re.shape[0]
    zc = z[..., :M].astype(np.float64) + 1j * z[..., M:].astype(np.float64)
    return zc @ np.conj(bf_re + 1j * bf_im)


# ---------------------------------------------------------------------------
# metrics (per clip, relative to the clip's largest reference value; the worst clip)
# ---------------------------------------------------------------------------
def rel_err(got, ref):
    got = np.asarray(got, np.float64).reshape(len(ref), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-300)
    return float((np.abs(got - ref).max(axis=1) / scale).max())


def f64_excess(got32, ref):
    """Error of float32-stored results beyond the rounding of the exact value to float32."""
    got = np.asarray(got32, np.float64)
    ex = np.abs(got - ref) - U32 * np.abs(ref)
    scale = np.maximum(np.abs(ref).max(axis=1), 1e-300)
    return float(max((ex.max(axis=1) / scale).max(), 0.0))


def report(label, **errs):
    print(f"[power-paths] {label}: " + ", ".join(f"{k}={v:.3e}" for k, v in errs.items()))


def check_doa(doa, p64, tol):
    """The first maximum of the reference; with a non-zero tolerance a column within `tol` of the maximum passes too
    (random steering: two columns closer than the float32 arithmetic are a near-tie, not a wrong index)."""
    want = first_argmax(p64)
    for b, d in enumerate(np.asarray(doa)):
        if d != want[b]:
            assert tol > 0 and 0 <= d < p64.shape[1] and p64[b, d] >= p64[b].max() * (1 - tol), (b, d, want[b])


# ---------------------------------------------------------------------------
# arrays and engines
# ---------------------------------------------------------------------------
BASE = "snn_c1_bipolar"          # STHT kernel, band, tau and RZCC width of every synthetic array below


def array_case(M, G, seed=0):
    """The base case on a circular array of M microphones (radius 4.5 cm) with a random float64 steering matrix: the
    quadratic form does not care what the steering vectors are."""
    g = dict(H.load(BASE))
    th = 2 * np.pi * np.arange(M) / M
    g["r_vec"], g["theta_vec"] = np.full(M, 4.5e-2), th
    g["x"] = np.zeros((1, M), np.float32)             # shape source of H.chain_spec
    g["bf_mat"] = np.random.default_rng(1000 * M + G + seed).standard_normal((2 * M, G))
    return g


def engine(g, T, bf=None):
    from haghighatshoarmuir2024_b200.engine import SnnEngine
    return SnnEngine(H.chain_spec(g, T), g["bf_mat"] if bf is None else bf, device=0)


def clips(g, B, T, seed, int16=False):
    return H.synth_clips(g, B, T, seed=seed, snrs_db=(-5.0, 5.0, 20.0), int16=int16)[0]


def to_dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def spec_membrane(eng, spikes):
    s = eng.spec
    return membrane64(spikes, s.neuron_decay, s.neuron_scale, s.neuron_len)


def chunk_bounds(G, C2, B, wide):
    """DoA slices of run_power: nchunk = min(ceil(SMs / B), ceil(G / 32)) when B < SMs and G C2^2 >= 2^20; slice
    length ceil(G / nchunk), rounded up to 32 for k_power_wide.  Returns the slice starts."""
    sms = sm_count()
    if not (B < sms and G * C2 * C2 >= (1 << 20)):
        return [0]
    nchunk = max(1, min((sms + B - 1) // B, (G + 31) // 32))
    gper = -(-G // nchunk)
    if wide:
        gper = (gper + 31) & ~31
    return list(range(0, G, gper))


@pytest.fixture(autouse=True, scope="module")
def _timing():
    t0 = time.perf_counter()
    yield
    print(f"\n[power-paths] test_gpu_power_paths.py: {time.perf_counter() - t0:.1f} s")


def _env(monkeypatch, env):
    for k in ("MICLOC_GRAM_FP32", "MICLOC_POWER_NARROW", "MICLOC_NO_SEGMENTS", "MICLOC_FUSED_FIR"):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


# ---------------------------------------------------------------------------
# a. membrane tap against membrane64 of the same call's spikes
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("B,T,segmented", [(2, 40_000, True), (3, 4_801, False)])
def test_membrane_tap_equals_the_float64_alpha_fir_of_its_spikes(B, T, segmented, monkeypatch):
    """k_neuron_seg: B = 2, T = 40 000 (few long clips: plan_segments cuts the neuron into segments of >= 1024 samples
    that start nwarm samples early, the warm-up path) and B = 3, T = 4 801 (one sequential segment)."""
    _env(monkeypatch, {})
    g = H.load(BASE)
    x = clips(g, B, T, seed=T)
    eng = engine(g, T)
    out = eng.run_taps(to_dev(x), want=("spikes", "vmem"))
    torch.cuda.synchronize()
    sp = out["spikes"].cpu().numpy()
    ref = spec_membrane(eng, sp)
    err = rel_err(out["vmem"].cpu().numpy(), ref)
    report(f"membrane B={B} T={T} segmented={segmented}", rel=err)
    assert np.count_nonzero(sp) > T // 100
    assert err < MEMBRANE_REL


# ---------------------------------------------------------------------------
# b. every Gram x power path against power64 of the call's own membrane
# ---------------------------------------------------------------------------
SMS = "SMS"          # placeholder: resolved to the device's SM count at run time

POWER_CASES = [
    # id, M, B, T, G, env, arithmetic of the Gram kernel (bound)
    ("gram-M1", 1, 3, 1025, 37, {}, "f64"),
    ("gram-M7-T255", 7, 4, 255, 64, {}, "f64"),
    ("gram-M7-T256", 7, 4, 256, 64, {}, "f64"),
    ("gram-M8-T1023", 8, 2, 1023, 100, {}, "f64"),
    ("gram-M7-B=SMs", 7, SMS, 1024, 449, {}, "f64"),
    ("gram-M7-B=SMs-1-chunked", 7, SMS + "-1", 1024, 5401, {}, "f64"),
    ("slab-M7-T70001", 7, 2, 70_001, 64, {}, "f64"),
    ("slab-M8-T65536", 8, 1, 65_536, 33, {}, "f64"),
    ("tiled-M16-T1024", 16, 3, 1024, 40, {}, "f32"),
    ("tiled-M16-wide-chunked", 16, 2, 1025, 1100, {}, "f32"),
    ("tiled-M16-narrow-chunked", 16, 2, 1025, 1100, {"MICLOC_POWER_NARROW": "1"}, "f32"),
    ("gram-M16-T20011-f64", 16, 1, 20_011, 1100, {"MICLOC_NO_SEGMENTS": "1"}, "f64"),
    ("tiled-M31-T20011", 31, 2, 20_011, 181, {}, "f32"),
    ("gram-M32-T255-wide", 32, 2, 255, 181, {}, "f64"),
    ("tc1-M32-wide-chunked", 32, 2, 1024, 256, {}, "tc"),
    ("tc1-M64-T20011", 64, 1, 20_011, 512, {}, "tc"),
    ("tiled1-M64-T20011", 64, 1, 20_011, 512, {"MICLOC_GRAM_FP32": "1"}, "f32"),
    ("tc1-M64-narrow", 64, 2, 3000, 200, {"MICLOC_POWER_NARROW": "1"}, "tc"),
    ("tc2-M72-wide-edge", 72, 1, 1024, 300, {}, "tc"),
    ("tc2-M73-narrow-smem", 73, 1, 1024, 300, {}, "tc"),
    ("tc2-M84-narrow-smem", 84, 2, 1025, 300, {}, "tc"),
    ("tc2-M85-narrow-global", 85, 1, 1024, 300, {}, "tc"),
    ("tc2-M96-T20011", 96, 3, 20_011, 300, {}, "tc"),
    ("gram-M96-f64-global", 96, 2, 3000, 300, {"MICLOC_NO_SEGMENTS": "1"}, "f64"),
    ("tc2-M128-T20011", 128, 1, 20_011, 512, {}, "tc"),
    ("tiled2-M128", 128, 2, 3000, 200, {"MICLOC_GRAM_FP32": "1"}, "f32"),
]


def _batch(B):
    if B == SMS:
        return sm_count()
    if B == SMS + "-1":
        return sm_count() - 1
    return B


@pytest.mark.parametrize("case", POWER_CASES, ids=[c[0] for c in POWER_CASES])
def test_every_gram_and_power_path_equals_power64_of_its_membrane(case, monkeypatch):
    """One row of the path table per case (see the module docstring):
      gram-*: k_gram + k_power_argmax<true> (C2 < 32; T = 255 / 256 around the tiled cut; B = SMs: one CTA per clip;
              B = SMs - 1 with G C2^2 >= 2^20: two DoA slices + k_argmax_chunks), or k_gram at C2 >= 32 when T < 256
              or MICLOC_NO_SEGMENTS (then k_power_wide at M = 16 / 32, k_power_argmax<false> at M = 96);
      slab-*: k_gram_slab + k_gram_reduce (C2 < 32, T >= 65536, few clips: 64 slabs);
      tiled-*: k_gram_tiled (M = 16, 31), tiled1 / tiled2: MICLOC_GRAM_FP32 at M = 64 (one 128 block) and M = 128
              (off-diagonal block);
      tc1-*: k_gram_tc<true> (M = 32, 64), tc2-*: k_gram_tc<false> (M = 72, 73, 84, 85, 96: second 128 tile half
              empty, 128: 2 x 2 blocks);
      power: k_power_wide for 32 <= C2 and M <= 72 (M = 72 is the 200 KB edge), chunked at G = 1100 (M = 16), 256
              (M = 32), 512, 300 (M >= 64, B < SMs); MICLOC_POWER_NARROW and M = 73, 84: k_power_argmax<true>;
              M = 85, 96, 128: k_power_argmax<false> (Gram read from global memory)."""
    label, M, B, T, G, env, kind = case
    _env(monkeypatch, env)
    B = _batch(B)
    g = array_case(M, G)
    x = clips(g, B, T, seed=M + T)
    eng = engine(g, T)
    out = eng.run_taps(to_dev(x), want=("vmem", "power", "doa"))
    torch.cuda.synchronize()
    p64 = power64(out["vmem"].cpu().numpy(), g["bf_mat"])
    p = out["power"].cpu().numpy()
    rel = rel_err(p, p64)
    ex = f64_excess(p, p64)
    report(label, rel=rel, f64_excess=ex)
    tol = {"f64": 0.0, "f32": F32_REL, "tc": TC_REL}[kind]
    if kind == "f64":
        assert ex < F64_EXCESS
    else:
        assert rel < tol
    assert rel < 32 / (10 * T)
    check_doa(out["doa"].cpu().numpy(), p64, tol)
    assert int(out["flags"].sum()) == 0


@pytest.mark.parametrize("M,G", [(7, 64), (8, 50), (16, 40)])
def test_dense_output_equals_the_float64_projection(M, G, monkeypatch):
    """k_dense<16> (C2 <= 16: M = 7, and M = 8 with all 16 weights in registers) and k_dense<0> (M = 16): `y` against
    the float64 product of the call's own membrane and bf_mat; G not a multiple of the 128-thread block, T of the
    256-sample slab."""
    _env(monkeypatch, {})
    g = array_case(M, G)
    T = 1000
    x = clips(g, 2, T, seed=3)
    eng = engine(g, T)
    out = eng.run_taps(to_dev(x), want=("vmem", "y"))
    torch.cuda.synchronize()
    ref = out["vmem"].cpu().numpy().astype(np.float64) @ g["bf_mat"]
    err = rel_err(out["y"].cpu().numpy(), ref)
    report(f"k_dense M={M}", rel=err)
    assert err < DENSE_REL


# ---------------------------------------------------------------------------
# c. first maximum: identical columns and planted ties
# ---------------------------------------------------------------------------
# id, M, B, T, G, env, k_power_wide
TIE_CASES = [
    ("argmax-M7", 7, 3, 1024, 64, {}, False),
    ("argmax-M7-chunked", 7, 2, 1024, 5401, {}, False),
    ("wide-M16", 16, 3, 1024, 40, {}, True),
    ("wide-M16-chunked", 16, 1, 1024, 1100, {}, True),
    ("narrow-M16-chunked", 16, 1, 1024, 1100, {"MICLOC_POWER_NARROW": "1"}, False),
    ("argmax-smem-M84-chunked", 84, 1, 1024, 300, {}, False),
    ("argmax-global-M96-chunked", 96, 2, 1024, 300, {}, False),
]


def _tie_pairs(bounds, G):
    """(a, b) with a < b: in different DoA slices (first slice / last slice, and two neighbouring slices at their
    seam) and inside one slice."""
    pairs = [(1, G - 2)]
    if len(bounds) > 1:
        s = bounds[1]
        pairs += [(s - 1, s), (bounds[0], bounds[-1]), (s, min(s + 5, G - 1))]
    else:
        pairs += [(0, 1), (G // 3, G // 2)]
    return pairs


@pytest.mark.parametrize("case", TIE_CASES, ids=[c[0] for c in TIE_CASES])
def test_staged_paths_return_the_first_maximum(case, monkeypatch):
    """k_power_argmax<true> (M = 7, 84; MICLOC_POWER_NARROW at M = 16), k_power_wide (M = 16) and
    k_power_argmax<false> (M = 96), with and without DoA slices (k_argmax_chunks: G = 5401 at M = 7, 1100 at M = 16,
    300 at M >= 84).  All columns equal -> DoA 0; two maximal columns w at a < b, every other column 0.5 w -> DoA a,
    with a and b in different slices (bounds computed as run_power does) and in one slice."""
    label, M, B, T, G, env, wide = case
    _env(monkeypatch, env)
    g = array_case(M, G)
    x = clips(g, B, T, seed=M)
    eng = engine(g, T)
    xd = to_dev(x)
    w = np.random.default_rng(M).standard_normal(2 * M)
    eng.set_bf(np.repeat(w[:, None], G, axis=1))
    out = eng.run_taps(xd, want=("power", "doa"))
    torch.cuda.synchronize()
    p = out["power"].cpu().numpy()
    assert (p == p[:, :1]).all() and out["doa"].tolist() == [0] * B, label
    bounds = chunk_bounds(G, 2 * M, B, wide)
    assert (len(bounds) > 1) == ("chunked" in label)
    for a, b in _tie_pairs(bounds, G):
        bf = np.repeat(0.5 * w[:, None], G, axis=1)
        bf[:, a] = bf[:, b] = w
        eng.set_bf(bf)
        out = eng.run_taps(xd, want=("power", "doa"))
        torch.cuda.synchronize()
        p = out["power"].cpu().numpy()
        assert (p[:, a] == p[:, b]).all() and (p[:, a] == p.max(axis=1)).all()
        assert out["doa"].tolist() == [a] * B, (label, a, b, bounds[:3])


@pytest.mark.parametrize("variant", ["tc", "ffma"])
@pytest.mark.parametrize("M", [7, 8])
def test_fused_and_beamformer_return_the_first_maximum(M, variant, monkeypatch):
    """Fused epilogues (specialised M = 7, generic M = 8) and the Hilbert beamformer's k_cpower_argmax: all columns
    equal -> DoA 0, two maximal columns a < b -> DoA a."""
    from haghighatshoarmuir2024_b200 import _native as N
    _env(monkeypatch, {"MICLOC_FUSED_FIR": "ffma"} if variant == "ffma" else {})
    G, T, B = 70, 2000, 4
    g = array_case(M, G)
    x = clips(g, B, T, seed=9)
    eng = engine(g, T)
    xd = to_dev(x)
    w = np.random.default_rng(M).standard_normal(2 * M)
    lib = N.lib()
    for a, b in ((0, 0), (3, 64), (31, 32)):
        bf = np.repeat((1.0 if a == b else 0.5) * w[:, None], G, axis=1)
        bf[:, a] = bf[:, b] = w
        eng.set_bf(bf)
        out = eng.run(xd, want_spikes=False, fused=True)
        torch.cuda.synchronize()
        assert not eng._fused_unsupported
        assert out["doa"].tolist() == [a] * B, (a, b)
        # beamformer: bf = w_re + i w_im per microphone
        re, im = np.ascontiguousarray(bf[:M]), np.ascontiguousarray(bf[M:])
        y = torch.empty((B, T, G, 2), dtype=torch.float32, device="cuda")
        doa = torch.empty(B, dtype=torch.int32, device="cuda")
        N.check(lib.micloc_hilbert_beamform(eng._h, C.c_void_p(xd.data_ptr()), N.F32, B, T, re.ctypes.data_as(N._dp),
                                            im.ctypes.data_as(N._dp), G, C.c_void_p(y.data_ptr()), None,
                                            C.c_void_p(doa.data_ptr()), None))
        torch.cuda.synchronize()
        assert doa.tolist() == [a] * B, (a, b)


# ---------------------------------------------------------------------------
# d. fused kernels against power64(membrane64(fused spikes))
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["tc", "ffma"])
@pytest.mark.parametrize("M", [2, 3, 8, "c2"])
def test_fused_power_equals_power64_of_the_fused_spikes(M, variant, monkeypatch):
    """Fused epilogues (tensor-core Gram, float64 quadratic form) of the generic-M instantiation at M = 2, 3 and 8
    (8 fills the 16-wide Gram tile), and the M = 7 instantiation on config 2 (one-second clips, G = 449 of band 1):
    power against power64(membrane64(spikes)) of the same call; with and without the spike output the same power and
    DoA."""
    _env(monkeypatch, {"MICLOC_FUSED_FIR": "ffma"} if variant == "ffma" else {})
    if M == "c2":
        g = H.load("full_c2_b1")
        T, B = 48_000, 4
        x = H.synth_clips(g, B, T, seed=12, snrs_db=(-5.0, 10.0))[0]
    else:
        g = array_case(M, 97)
        T, B = 4_801, 12
        x = clips(g, B, T, seed=M)
    eng = engine(g, T)
    xd = to_dev(x)
    out = eng.run(xd, want_spikes=True, fused=True)
    bare = eng.run(xd, want_spikes=False, fused=True)
    torch.cuda.synchronize()
    assert not eng._fused_unsupported and int(out["flags"].sum()) == 0
    p64 = power64(spec_membrane(eng, out["spikes"].cpu().numpy()), g["bf_mat"])
    p = out["power"].cpu().numpy()
    err = rel_err(p, p64)
    report(f"fused {variant} M={M}", rel=err)
    assert err < FUSED_REL and err < 32 / (10 * T)
    check_doa(out["doa"].cpu().numpy(), p64, FUSED_REL)
    assert torch.equal(bare["power"], out["power"]) and torch.equal(bare["doa"], out["doa"])


# ---------------------------------------------------------------------------
# e. micloc_snn_gram
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("int16", [False, True])
@pytest.mark.parametrize("M", [7, 16, 64])
def test_design_gram_equals_gram64_from_t_start(M, int16, monkeypatch):
    """micloc_snn_gram (sequential front end + k_gram with t_start > 0), B = 3: against gram64 of the same front
    end's membrane tap from t_start (float64 sums: 1e-12) and of membrane64 of its spikes (float32 membrane);
    t_start in {0, 1, T // 4, T - 1}; symmetric; t_start = T and t_start < 0 rejected."""
    _env(monkeypatch, {"MICLOC_NO_SEGMENTS": "1"})
    g = array_case(M, 24)
    T, B = 3001, 3
    x = clips(g, B, T, seed=M, int16=int16)
    eng = engine(g, T)
    xd = to_dev(x)
    tap = eng.run_taps(xd, want=("spikes", "vmem"))
    torch.cuda.synchronize()
    vm = tap["vmem"].cpu().numpy()
    v64 = spec_membrane(eng, tap["spikes"].cpu().numpy())
    worst = worst_m = 0.0
    for t0 in (0, 1, T // 4, T - 1):
        gd = eng.gram(xd, t0)
        torch.cuda.synchronize()
        gm = gd.cpu().numpy()
        assert np.array_equal(gm, np.swapaxes(gm, 1, 2)), t0
        e = rel_err(gm, gram64(vm, t0))
        em = rel_err(gm, gram64(v64, t0))
        worst, worst_m = max(worst, e), max(worst_m, em)
        assert e < F64_EXCESS, t0
        assert em < MEMBRANE_REL, t0
    report(f"gram M={M} int16={int16}", f64=worst, vs_membrane64=worst_m)
    for bad in (T, -1):
        with pytest.raises(ValueError):
            eng.gram(xd, bad)


# ---------------------------------------------------------------------------
# f. micloc_hilbert_beamform through the C ABI
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("int16", [False, True])
@pytest.mark.parametrize("M", [7, 16])
def test_hilbert_beamform_equals_cproject64_of_its_band_pass(M, int16, monkeypatch):
    """micloc_hilbert_beamform: k_cproject (`y`) against cproject64 of the `z` tap of run_taps on the same context
    and input, k_cpower_argmax (power, DoA) against mean |y|^2 of the device's y (float64 sums) and of y64.
    B = 3, M = 7 (float32 FIR) and 16 (tensor-core STHT), T = 3001, G = 200."""
    from haghighatshoarmuir2024_b200 import _native as N
    _env(monkeypatch, {})
    G, T, B = 200, 3001, 3
    g = array_case(M, G)
    x = clips(g, B, T, seed=M + 1, int16=int16)
    eng = engine(g, T)
    xd = to_dev(x)
    rng = np.random.default_rng(M)
    bf_re, bf_im = rng.standard_normal((M, G)), rng.standard_normal((M, G))
    y = torch.empty((B, T, G, 2), dtype=torch.float32, device="cuda")
    power = torch.empty((B, G), dtype=torch.float32, device="cuda")
    doa = torch.empty(B, dtype=torch.int32, device="cuda")
    ptr = lambda t: C.c_void_p(t.data_ptr())
    lib = N.lib()
    N.check(lib.micloc_hilbert_beamform(eng._h, ptr(xd), N.I16 if int16 else N.F32, B, T, bf_re.ctypes.data_as(N._dp),
                                        bf_im.ctypes.data_as(N._dp), G, ptr(y), ptr(power), ptr(doa), None))
    z = eng.run_taps(xd, want=("z",))["z"]
    torch.cuda.synchronize()
    yd = y.cpu().numpy()
    yc = yd[..., 0].astype(np.float64) + 1j * yd[..., 1].astype(np.float64)
    y64 = cproject64(z.cpu().numpy(), bf_re, bf_im)
    ey = rel_err(yc, y64)
    pd = np.mean(np.abs(yc) ** 2, axis=1)
    p64 = np.mean(np.abs(y64) ** 2, axis=1)
    p = power.cpu().numpy()
    ex = f64_excess(p, pd)
    ep = rel_err(p, p64)
    report(f"hilbert M={M} int16={int16}", y=ey, power_f64_excess=ex, power_vs_y64=ep)
    assert ey < DENSE_REL
    assert ex < F64_EXCESS
    assert ep < DENSE_REL
    check_doa(doa.cpu().numpy(), pd, 0.0)
    check_doa(doa.cpu().numpy(), p64, DENSE_REL)


# ---------------------------------------------------------------------------
# g. stream batch power on a wide array
# ---------------------------------------------------------------------------
def test_stream_batch_power_on_96_microphones():
    """Stream batches share launch_power with run_taps: at M = 96 (k_power_argmax<false>, per-slot row counts) one
    push of 3 slots against power64 of membrane64 of each slot's final spikes."""
    from haghighatshoarmuir2024_b200.engine import SnnStreamBatch
    M, G, S, n = 96, 150, 3, 4000
    g = array_case(M, G)
    x = clips(g, S, n, seed=96)
    eng = engine(g, n)
    sb = SnnStreamBatch(eng, S, max_frame_len=n)
    out = sb.push(to_dev(x))
    torch.cuda.synchronize()
    rows = out["n_out"]
    assert rows.tolist() == [n - sb.latency] * S
    sp = out["spikes"].cpu().numpy()
    p64 = np.stack([power64(spec_membrane(eng, sp[s, :rows[s]])[None], g["bf_mat"])[0] for s in range(S)])
    p = out["power"].cpu().numpy()
    err = rel_err(p, p64)
    report("stream batch M=96", rel=err)
    assert err < MEMBRANE_REL
    check_doa(out["doa"].cpu().numpy(), p64, MEMBRANE_REL)
    sb.close()
