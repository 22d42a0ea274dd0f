#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native micloc SNN-localisation hot path.

Workload (BASELINE.json configs[1]): the Monte-Carlo SNR sweep of
paper_plots/target_snn_localization.py on a 7-microphone centre-circular array
(r = 4.5 cm), fs = 48 kHz, 1 s clips, 10 ms STHT kernel, bipolar RZCC, 449-angle DoA
grid, the three bands 1600-2000 / 2000-2300 / 2300-2600 Hz, 11 SNRs in [-10, 20] dB.
One STEP = one batch of `--clips-per-band` clips for each of the three bands through
the fused STHT -> band-pass -> RZCC -> neuron filter -> beamforming power -> argmax
kernel (3 launches), plus the DoA histogram (and its NCCL all-reduce when N > 1).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N
    python bench.py --impl reference ...        # the CPU path on the host cores
    python bench.py ... --dump-outputs DIR      # + what the last timed step returned, as DIR/<name>.npy

Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

FS = 48_000
T_CLIP = 48_000
NUM_MIC = 7
SNR_GRID = np.linspace(-10, 20, 11)          # target_snn_localization.py:435
METRIC = "clips_per_sec"
UNIT = "clips/s"
RHO_NOMINAL = 0.076                          # spikes per channel-sample (SURVEY.md 8d); measured value is reported
DUMP_BYTES_MAX = 64 << 20
DUMP_SPIKE_CLIPS = 4                         # spike rasters are [B, T, 14] int8 per band (4.8 GB at the default B)


def dump_outputs(out_dir, outs, hist=None):
    """Write what one step returned to its caller as <out_dir>/<name>.npy: per band `b`, `<key>_band<b>` for every array
    of the band's result (DoA index and RZCC flags of every clip as float32), the spike rasters of a fixed, seeded
    sample of clips as float32 (`spikes_band<b>_clips` holds their indices), and the step's DoA histogram as float64.
    The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    arrays = {}
    for b, out in enumerate(outs):
        for key, v in out.items():
            if not hasattr(v, "shape"):
                continue
            if key == "spikes":
                rows = np.sort(np.random.default_rng(0).choice(len(v), min(DUMP_SPIKE_CLIPS, len(v)), replace=False))
                arrays[f"spikes_band{b}_clips"] = rows.astype(np.float64)
                v = v[rows.tolist()]
            v = v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)
            arrays[f"{key}_band{b}"] = v.astype(np.float64 if v.dtype == np.float64 else np.float32)
    if hist is not None:
        arrays["doa_histogram"] = hist.cpu().numpy().astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES_MAX:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_BYTES_MAX}; use fewer clips per band")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_workload():
    d = np.load(os.path.join(ROOT, "tests", "golden", "bench_c2_bf.npz"))
    bands = [list(map(float, b)) for b in d["bands"]]
    return d, bands


def flops_per_mic_sample(K, M, G, rho, gram=True):
    """Algorithmic FLOP per microphone sample (FMA = 2), DESIGN.md 'Roofline'.
    survey: F = K + 40 + G (2 rho + 6/M)                       (SURVEY.md 8d; per-neuron time loop)
    gram  : F = K + 40 + 24 + (2M)(2M+1)/M                      (what the fused kernel has to do:
            240 FMA STHT, 2 ch x 2 biquads x 9, cumsum/sign, 2 ch x 12 neuron, upper-triangular Gram)"""
    if gram:
        return K + 40 + 24 + (2 * M) * (2 * M + 1) / M
    return K + 40 + G * (2 * rho + 6.0 / M)


# --------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# --------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores
# --------------------------------------------------------------------------------------
def host_clips(d, band_idx, bands, n, seed):
    """n clips of band `band_idx` synthesised on the HOST with numpy (same recipe as
    SnrSweep.synthesize / SNNBeamformer.apply_to_template)."""
    rng = np.random.default_rng(seed)
    band = bands[band_idx]
    t = np.arange(T_CLIP) / FS
    f0 = band[1]
    r, th = d["r_vec"], d["theta_vec"]
    corr = 10 * np.log10((FS / 2) / (band[1] - band[0]))
    xs = np.empty((n, T_CLIP, NUM_MIC), dtype=np.float32)
    for i in range(n):
        doa = rng.uniform(0, 2 * np.pi)
        dl = -r * np.cos(th - doa) / 340.0
        dl = dl - dl.min()
        td = t[None, :] - dl[:, None]
        td[td < 0] = 0
        x = np.interp(td.ravel(), t, np.sin(2 * np.pi * f0 * t)).reshape(td.shape).T
        snr = 10 ** ((SNR_GRID[i % len(SNR_GRID)] - corr) / 10)
        xs[i] = x + np.sqrt(np.mean(x ** 2)) / np.sqrt(snr) * rng.standard_normal(x.shape)
    return xs


def oracle_cfgs(d, bands):
    from scipy.signal import butter
    from oracle import oracle as O
    cfgs = []
    t = np.arange(T_CLIP) / FS
    for i, band in enumerate(bands):
        b, a = butter(2, band, btype="bandpass", analog=False, output="ba", fs=FS)
        tau = float(d[f"tau_{i}"])
        cfgs.append(O.SnnConfig(h=d["kernel"], b=b, a=a, robust_width=float(d[f"robust_width_{i}"]), bipolar=True,
                                nir=O.neuron_kernel(t, tau, tau), bf=d[f"bf_{i}"]))
    return cfgs


def cpu_pass(cfgs, clips_per_band, nthreads):
    """One bounded pass of the CPU path: sum over bands of (clips, seconds)."""
    from oracle import oracle as O
    t0 = time.perf_counter()
    n = 0
    outs = []
    for cfg, x in zip(cfgs, clips_per_band):
        outs.append(O.snn_run_batch(cfg, x, nthreads=nthreads, want_power=False, want_spikes=False))
        n += x.shape[0]
    return n, time.perf_counter() - t0, outs


def reference_python(n_per_band=0):
    """The unmodified reference Python beside the port (BASELINE.md section 3: multiprocessing.Pool over the host
    cores): timed live when /root/reference is importable (build container), else the committed measurement of
    tools/time_reference_python.py -- the GPU box has no /root/reference."""
    if os.path.isdir("/root/reference") and n_per_band > 0:
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import time_reference_python as TR
            v, doa, _, secs, cores = TR.time_reference(n_per_band)
            return {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "measured": "live",
                    "sample": f"{len(doa)} clips in {secs:.1f} s, multiprocessing.Pool({cores})"}
        except Exception as e:
            return {"unavailable": f"{type(e).__name__}: {e}"}
    f = os.path.join(ROOT, "profiles", "r02_reference_python_timing.json")
    if os.path.exists(f):
        j = json.load(open(f))
        return {"value": j["reference_python_clips_per_s"], "unit": UNIT, "cores": j["cores"], "kind": "reference",
                "measured": "committed (profiles/r02_reference_python_timing.json): " + j["where"],
                "oracle_port_same_host": j["oracle_port_clips_per_s_same_host"], "port_over_python": j["port_over_python"],
                "doa_identical_port_vs_python": j["doa_identical_port_vs_python"]}
    return {"unavailable": "no /root/reference on this host and no committed measurement"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    d, bands = load_workload()
    cores = os.cpu_count() or 1
    cfgs = oracle_cfgs(d, bands)
    n_per_band = cores if args.cpu_clips_per_band <= 0 else args.cpu_clips_per_band
    clips = [host_clips(d, i, bands, n_per_band, seed=1000 + i) for i in range(len(bands))]
    for _ in range(args.warmup):
        cpu_pass(cfgs, [c[:1] for c in clips], cores)
    tot_n, tot_s = 0, 0.0
    for _ in range(args.steps):
        n, s, outs = cpu_pass(cfgs, clips, cores)
        tot_n += n; tot_s += s
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs)
    v = tot_n / tot_s
    sample = f"{n_per_band} clips x {len(bands)} bands per step (1 s, 7 mics, G=449), {args.steps} steps"
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(n_per_band, "f32"),
        "mic_msamples_per_sec": v * T_CLIP * NUM_MIC / 1e6,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "oracle/micloc_oracle.c: C restatement of SNNBeamformer.apply_to_signal + power/argmax, "
                                 "pinned bit-identical to numpy/scipy on tests/golden; pthreads over clips",
                         "reference_python": reference_python(max(2, n_per_band // 4))},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def workload_config(clips_per_band, dtype):
    return {"workload": "configs[1]: Monte-Carlo SNR sweep (target_snn_localization.py), 7-mic centre-circular array "
                        "r=4.5cm, fs=48kHz, 1 s clips, bands 1600-2000/2000-2300/2300-2600 Hz, G=449, bipolar RZCC, "
                        "11 SNRs -10..20 dB, random DoA",
            "clips_per_band_per_step": clips_per_band, "bands": 3, "clip_samples": T_CLIP, "num_mic": NUM_MIC,
            "num_doa": 449, "stht_taps": 480, "input_dtype": dtype,
            "cache": "per-step input >> 126 MB L2 (no flush needed)", "parallelism": "clips sharded by rank"}


# --------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist

    from haghighatshoarmuir2024_b200 import _native as N
    from haghighatshoarmuir2024_b200.montecarlo import BandSetup, SnrSweep

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # pin this rank (and the pinned staging it allocates from now on) to its GPU's NUMA node: the host-buffer leg
    # streams tens of GB/s per GPU over PCIe
    from haghighatshoarmuir2024_b200.distributed import bind_to_gpu_numa
    numa = bind_to_gpu_numa(local, int(os.environ.get("LOCAL_WORLD_SIZE", world)))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = N.lib()

    d, bands = load_workload()
    nb = len(bands)
    Bb = args.clips_per_band
    tdtype = torch.int16 if args.dtype == "i16" else torch.float32
    setups = [BandSetup(band=bands[i], tau=float(d[f"tau_{i}"]), bf_mat=d[f"bf_{i}"]) for i in range(nb)]
    sweep = SnrSweep(setups, d["r_vec"], d["theta_vec"], FS, float(d["kernel_duration"]), T_CLIP, device=local)
    G = sweep.G
    audio, doa_true = [], []
    for i in range(nb):
        a, dt_, _ = sweep.synthesize(i, Bb, seed=10_000 * (rank + 1) + i, snr_db_grid=SNR_GRID, dtype=tdtype)
        audio.append(a); doa_true.append(dt_)
    torch.cuda.synchronize()
    hist = torch.zeros(G, dtype=torch.int64, device=dev)
    # one stream per band: the three fused launches of a step are independent, so the tail of one
    # (persistent CTAs running out of clip pairs) overlaps the head of the next
    side = [torch.cuda.Stream(device=dev) for _ in range(nb)] if args.band_streams else None

    refined = [0]

    def step(want_spikes=True):
        hist.zero_()
        outs = []
        cur = torch.cuda.current_stream(dev)
        for i in range(nb):
            if side:
                side[i].wait_stream(cur)
                with torch.cuda.stream(side[i]):
                    outs.append(sweep.run_band(i, audio[i], want_spikes=want_spikes, want_power=False, hist=None, refine=False))
            else:
                outs.append(sweep.run_band(i, audio[i], want_spikes=want_spikes, want_power=False, hist=None, refine=False))
        for i in range(nb):
            if side:
                cur.wait_stream(side[i])
            # clips the fused kernel's bounded RZCC encoder gave up on are redone by the library (flag read-back + sync,
            # inside the timed region; none on this workload)
            refined[0] += sweep.engines[i].refine(audio[i], outs[i])
            sweep.histogram(outs[i]["doa"], hist)
        if world > 1:
            dist.all_reduce(hist)          # the only cross-GPU exchange: DoA histograms (SURVEY.md 8e)
        return outs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput (`value`) ----
    for _ in range(args.warmup):
        outs = step()
    barrier()
    for e in sweep.engines:
        e.enable_timing(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = lib.micloc_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        outs = step()
    ev1.record()
    barrier()
    launches = lib.micloc_launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    kern_ms, kern_n = 0.0, 0
    for e in sweep.engines:
        m_, n_ = e.last_kernel_ms()
        kern_ms += m_; kern_n += n_
        e.enable_timing(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs, hist)
    # cross-check of the launch time with one launch at a time (no overlap between the bands): the library's CUDA events
    # around every k_fused_tc launch on its stream, two passes over the three bands, outside the timed region
    solo_ms, solo_n = 0.0, 0
    for e in sweep.engines:
        e.enable_timing(True)
    for _ in range(2):
        for i in range(nb):
            o_ = sweep.run_band(i, audio[i], want_spikes=True, want_power=False, hist=None, refine=False)
            torch.cuda.synchronize()
            del o_
    for e in sweep.engines:
        m_, n_ = e.last_kernel_ms()
        solo_ms += m_; solo_n += n_
        e.enable_timing(False)
    tm = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_max = float(tm.item())
    clips_step_all = nb * Bb * world
    value = clips_step_all * args.steps / (ms_max * 1e-3)
    spike_density = float(np.mean([float(o["spikes"][:64].ne(0).float().mean()) for o in outs]))
    flags = int(sum(int(o["flags"].sum()) for o in outs))
    del outs
    torch.cuda.empty_cache()

    # ---- end to end through the C-ABI with HOST buffers (`e2e`): both wire formats ----
    # int16 PCM is the reference's wire format (micloc/record.py:54-75 reads integer wav frames) and the documented
    # default of the host path: half the PCIe bytes of float32.  `e2e` is the int16 leg, `e2e.f32` the float32 one.
    Be = min(Bb, args.e2e_clips_per_band)                          # bounded: the host copy of the full step would be tens of GB
    d2h = nb * Be * (4 + 4)                                       # doa + flags per clip

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(max_workers=nb)

    def e2e_leg(host):
        h2d = sum(h.numel() for h in host) * host[0].element_size()
        def e2e_step():
            # one host thread per band (ctypes drops the GIL inside the call): the bands are independent contexts with
            # their own staging streams, so the drain of one band's last chunk overlaps the next band's copies
            futs = [pool.submit(sweep.engines[i].run_host, host[i], False, False, True) for i in range(nb)]
            return [f.result() for f in futs]
        for _ in range(max(1, min(args.warmup, 2))):
            res = e2e_step()
        barrier()
        l1 = lib.micloc_launch_count()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = e2e_step()
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        n_launch = lib.micloc_launch_count() - l1
        te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        secs = float(te.item())
        return res, nb * Be * world * args.steps / secs, h2d, h2d * args.steps / secs / 1e9, n_launch

    host_f32 = [a[:Be].cpu().pin_memory() for a in audio] if tdtype == torch.float32 else None
    if tdtype == torch.int16:
        audio16 = audio
    else:
        audio16 = [sweep.synthesize(i, Be, seed=10_000 * (rank + 1) + i, snr_db_grid=SNR_GRID, dtype=torch.int16)[0]
                   for i in range(nb)]
    host_i16 = [a[:Be].cpu().pin_memory() for a in audio16]
    res16, e2e_value, h2d, e2e_gbs, nl = e2e_leg(host_i16)
    launches += nl
    # the host path and the device path must agree bit for bit
    dev_doa16 = [sweep.run_band(i, audio16[i][:Be], want_power=False)["doa"].cpu().numpy() for i in range(nb)]
    e2e_same = all(np.array_equal(res16[i]["doa"].numpy(), dev_doa16[i]) for i in range(nb))
    e2e_f32 = None
    dev_doa = [sweep.run_band(i, audio[i][:Be], want_power=False)["doa"].cpu().numpy() for i in range(nb)]
    host = host_f32 if host_f32 is not None else host_i16
    if host_f32 is not None:
        res32, v32, h2d32, gbs32, nl = e2e_leg(host_f32)
        launches += nl
        same32 = all(np.array_equal(res32[i]["doa"].numpy(), dev_doa[i]) for i in range(nb))
        e2e_f32 = {"value": v32, "unit": UNIT, "h2d_bytes_per_step": h2d32, "d2h_bytes_per_step": d2h,
                   "pcie_h2d_gbs": gbs32, "matches_device_path": bool(same32)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant (fused) kernel ----
    K = len(d["kernel"])
    mic_samples_per_launch = Bb * T_CLIP * NUM_MIC
    avg_launch_ms = kern_ms / max(kern_n, 1)
    F_gram = flops_per_mic_sample(K, NUM_MIC, G, spike_density, gram=True)
    F_survey = flops_per_mic_sample(K, NUM_MIC, G, spike_density, gram=False)
    if side:
        # the launches of a step overlap on the device: their individual event durations double-count shared
        # time, so the kernel time of a step is the step's own device time (the fused launches are all of it
        # but the three histogram launches, < 0.1 %)
        avg_launch_ms = (ms / args.steps) / nb
    achieved = mic_samples_per_launch * F_gram / (avg_launch_ms * 1e-3) / 1e12
    peak = {}
    for name, variant in (("ffma", 0), ("ffma2", 1)):
        import ctypes
        v = ctypes.c_double()
        N.check(lib.micloc_fp32_peak(local, variant, ctypes.byref(v)))
        peak[name] = v.value
    fp32_peak = max(peak.values())
    peaks_file = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_peak, hbm_src = 6650.0, "fallback"
    if os.path.exists(peaks_file):
        try:
            hbm_peak, hbm_src = float(json.load(open(peaks_file))["hbm_gbs"]), "measured"
        except Exception:
            pass
    in_bytes = 2 if args.dtype == "i16" else 4
    hbm_gbs = mic_samples_per_launch * (in_bytes + 2) / (avg_launch_ms * 1e-3) / 1e9
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "fused_traffic.json")
    if os.path.exists(tfile):
        try:
            tj = json.load(open(tfile))        # dram__bytes_read + write of one `ncu --set full` capture, per clip
            if args.dtype == tj.get("input_dtype", "f32"):
                traffic = float(tj["dram_bytes_per_clip"]) * Bb          # bytes per launch of Bb clips
        except Exception:
            pass
    # what the tensor cores execute for the STHT share (k_fused_tc): per tile of 128 stream samples x 32 columns a dense
    # 128 x 368 Toeplitz product in three fp16 pieces -- 2 x 3 x 128 x 368 x 32 FLOP for 2 clips x 256 frames x M microphones
    tensor_peak, tensor_src = 2250.0, "nominal dense fp16"
    try:
        tensor_peak, tensor_src = float(json.load(open(peaks_file))["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        pass
    mma_flop_per_mic_sample = 2.0 * 3 * 128 * 368 * 32 / (2 * 256 * NUM_MIC)
    tensor_tflops = mic_samples_per_launch * mma_flop_per_mic_sample / (avg_launch_ms * 1e-3) / 1e12
    roofline = {
        "bound": "fp32", "kernel": "k_fused" if os.environ.get("MICLOC_FUSED_FIR", "")[:1] == "f" else "k_fused_tc",
        "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
        "frac": achieved / fp32_peak, "traffic": traffic,
        "peak_source": f"measured in this run by micloc_fp32_peak (FFMA {peak['ffma']:.1f}, FFMA2 {peak['ffma2']:.1f} TFLOP/s)",
        "flop_per_mic_sample": F_gram, "flop_per_mic_sample_survey_formula": F_survey,
        "achieved_survey_formula": achieved * F_survey / F_gram,
        "note": "algorithmic FLOPs of the chain (574 per mic-sample, STHT = 480 of them) over the measured FP32 FMA peak, the "
                "north star's roofline; k_fused_tc executes the STHT share as fp16 hi/lo tcgen05.mma (3 products, 128x368 "
                "Toeplitz tiles), so the FP32 pipe itself carries only the 94 non-STHT FLOPs per mic-sample",
        "avg_launch_ms": avg_launch_ms, "launches_timed": kern_n, "mic_samples_per_launch": mic_samples_per_launch,
        "kernel_share_of_step": kern_ms / ms,
        "solo_launch_ms": solo_ms / max(solo_n, 1), "solo_launches_timed": solo_n,
        "solo_frac": (mic_samples_per_launch * F_gram / (solo_ms / max(solo_n, 1) * 1e-3) / 1e12) / fp32_peak,
        "launch_timing": ("3 band launches per step overlap on 3 streams: avg_launch_ms = step device time / 3; "
                          "kernel_share_of_step sums the overlapping per-launch event durations (> 1 when they overlap); "
                          "solo_launch_ms = CUDA events around single launches with nothing else running (their tails do not overlap)"
                          if side else "CUDA events around every launch on its stream, inside the library"),
        "tensor_view": {"achieved": tensor_tflops, "peak": tensor_peak, "unit": "TFLOP/s", "frac": tensor_tflops / tensor_peak,
                        "executed_flop_per_mic_sample": mma_flop_per_mic_sample, "peak_source": tensor_src,
                        "note": "fp16 tcgen05.mma FLOPs k_fused_tc executes for the STHT (dense Toeplitz tiles incl. their zeros, "
                                "hi/lo split x3): 5.3 x the 480 algorithmic FLOPs; not the bound"},
        "hbm_view": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                     "peak_source": hbm_src + " (MEASURED_PEAKS.json hbm_gbs)" if hbm_src == "measured" else "fallback 6650",
                     "bytes_per_mic_sample": in_bytes + 2},
    }

    # ---- CPU baseline beside it (rank 0, N == 1) + DoA match rate of the GPU path against it ----
    cpu = None
    match = None
    if world == 1 and not args.no_cpu:
        cores = os.cpu_count() or 1
        cfgs = oracle_cfgs(d, bands)
        n_cpu = args.cpu_clips_per_band if args.cpu_clips_per_band > 0 else 4 * cores      # ~4 s of wall time on all cores
        n_cpu = min(n_cpu, Bb, Be)
        xs = [host[i][:n_cpu].numpy() for i in range(nb)]
        n, s, ref = cpu_pass(cfgs, xs, cores)
        cpu = {"value": n / s, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"first {n_cpu} clips of each band of the GPU batch ({n} clips, {s:.1f} s wall)",
               "reference_python": reference_python(0)}
        same = np.concatenate([dev_doa[i][:n_cpu] == ref[i]["doa"] for i in range(nb)])
        match = {"doa_match_rate_vs_cpu_path": float(same.mean()), "clips_compared": int(same.size)}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(Bb, args.dtype),
        "mic_msamples_per_sec": value * T_CLIP * NUM_MIC / 1e6,
        "outputs_in_timed_region": "int8 spikes [B,T,14] + int32 DoA [B] + DoA histogram written to HBM",
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "micloc_snn_run_host (pinned host audio in, DoA indices + flags out), one host thread per band",
                "wire_format": "int16 PCM [B][T][M] (the reference's recorder format, micloc/record.py:54-75); "
                               "the float32 leg is under `f32`",
                "clips_per_band_per_step": Be, "pcie_h2d_gbs": e2e_gbs,
                "matches_device_path": bool(e2e_same), "f32": e2e_f32, "numa": numa},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "spike_density": spike_density, "rzcc_overflow_clips": flags, "rzcc_refined_clips": refined[0],
    }
    if world == 1 and not args.no_extras:
        del audio, audio16, host_i16, host_f32, host
        torch.cuda.empty_cache()
        try:
            line["configs"] = run_extras(args, local, fp32_peak, lib)
        except Exception as e:                                  # the headline line must not die with an extra
            import traceback
            line["configs"] = {"error": f"{type(e).__name__}: {e}", "trace": traceback.format_exc()[-1500:]}
    if cpu:
        line["cpu_baseline"] = cpu
    if match:
        line["parity"] = match
    emit(line)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------
# the other BASELINE configs (reported beside the headline line under "configs"; bounded to a few seconds each)
# --------------------------------------------------------------------------------------
def _timed(torch, fn, n=3):
    out = fn()
    out = fn()                     # twice: the caching allocator needs two generations of the output buffers
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, out


def run_extras(args, local, fp32_peak, lib):
    """Throughput + parity sample of BASELINE configs 1, 3, 4, 5 on this GPU (rank 0, N = 1).  Each entry: the call a
    user makes through the C-ABI, CUDA-event time over 3 runs after a warm-up, the roofline that bounds it, and a small
    sample of the same clips through the oracle.  Inputs are synthesised by the library's own kernels."""
    import ctypes
    import torch
    import helpers as H
    from oracle import oracle as O
    from haghighatshoarmuir2024_b200.engine import SnnEngine
    from haghighatshoarmuir2024_b200.montecarlo import synthesize_clips

    res = {}
    cores = os.cpu_count() or 1
    T = T_CLIP
    t = np.arange(T) / FS
    rng = np.random.default_rng(5)

    def fp32_entry(name, g, x, n_cmp, fused=True, what=""):
        M = x.shape[2]
        eng = SnnEngine(H.chain_spec(g, x.shape[1]), g["bf_mat"], device=local)
        l0 = lib.micloc_launch_count()
        ms, out = _timed(torch, lambda: eng.run(x, want_spikes=True, want_power=True, fused=fused))
        launches = (lib.micloc_launch_count() - l0) // 4
        B = x.shape[0]
        F = flops_per_mic_sample(len(g["kernel"]), M, g["bf_mat"].shape[1], 0.0, gram=True)
        ach = B * x.shape[1] * M * F / (ms * 1e-3) / 1e12
        parity = cpu_port = None
        if n_cmp:
            cfg = H.oracle_cfg(g)
            cfg.nir = O.neuron_kernel(np.arange(x.shape[1]) / FS, float(g["tau"]), float(g["tau"]))
            xc = x[:n_cmp].cpu().numpy()
            t0 = time.perf_counter()
            ref = O.snn_run_batch(cfg, xc, nthreads=min(cores, n_cmp), want_spikes=True)
            cpu_s = time.perf_counter() - t0
            doa = out["doa"][:n_cmp].cpu().numpy()
            parity = {"clips_compared": n_cmp, "doa_match_rate_vs_cpu_path": float((doa == ref["doa"]).mean()),
                      "spike_agreement": H.spike_agreement(out["spikes"][:n_cmp].cpu().numpy(), ref["spikes"]),
                      "power_rel_err": H.rel_err(out["power"][:n_cmp].cpu().numpy(), ref["power"])}
            cpu_port = {"clips_per_sec": n_cmp / cpu_s, "cores": min(cores, n_cmp)}
        res[name] = {
            "workload": what, "clips": B, "clip_samples": int(x.shape[1]), "num_mic": M, "num_doa": int(g["bf_mat"].shape[1]),
            "path": "fused k_fused_tc (1 launch)" if fused and not eng._fused_unsupported else
                    f"staged kernels: tensor-core STHT / Gram for wide arrays, time-segmented chains for long clips ({launches} launches)",
            "ms": ms, "clips_per_sec": B / ms * 1e3, "mic_msamples_per_sec": B * x.shape[1] * M / ms / 1e3,
            "roofline": {"bound": "fp32", "flop_per_mic_sample": F, "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": ach / fp32_peak},
            "parity": parity, "cpu_port": cpu_port,
            "rzcc_overflow_clips": int(out["flags"].sum()),
        }
        eng.close()

    # configs[0]: noisy wideband clips (in-band chirp + AWGN), 64-angle grid -- the reference's own CPU case, batched
    g = H.load("snn_c1_bipolar")
    B = args.extra_clips
    f_lo, f_hi = map(float, g["band"])
    chirp = np.sin(2 * np.pi * np.cumsum(f_lo + (f_hi - f_lo) * t / t[-1]) / FS)
    snr = 10 ** ((SNR_GRID[np.arange(B) % len(SNR_GRID)] - 10 * np.log10((FS / 2) / (f_hi - f_lo))) / 10)
    x = synthesize_clips(g["r_vec"], g["theta_vec"], FS, T, rng.uniform(0, 2 * np.pi, B), snr_lin=snr, source=chirp,
                         mode=0, seed=71, device=local)
    fp32_entry("c1", g, x, 16, what="configs[0] batched: 1 s noisy wideband (chirp 1600-2000 Hz + AWGN, 11 SNRs) clips, "
                                    "7-mic circular array, G=64, bipolar")
    del x

    # configs[3]: two simultaneous speech-shaped sources (band-limited coloured noise), 360-angle grid
    g = H.load("snn_c4_multi")
    from scipy.signal import butter, lfilter
    b_, a_ = butter(2, g["band"], btype="bandpass", fs=FS)
    S = 8
    src = np.stack([lfilter(b_, a_, lfilter([1.0], [1.0, -0.95], rng.standard_normal(T))) for _ in range(S)])
    doa2 = np.stack([rng.uniform(0, 2 * np.pi, B), rng.uniform(0, 2 * np.pi, B)], axis=1)
    x = synthesize_clips(g["r_vec"], g["theta_vec"], FS, T, doa2, snr_lin=np.full(B, 100.0), source=src,
                         source_index=np.arange(B) % S, gain=np.tile([1.0, 0.7], (B, 1)), mode=1, seed=72, device=local)
    fp32_entry("c4", g, x, 16, what="configs[3]: 1 s clips of two simultaneous speech-shaped sources "
                                    "(signal_multiple_targets), 7-mic array, G=360")
    del x

    # configs[4]: 64 microphones, 10 s clips, 512-angle grid (staged time-segmented kernels); parity on a 1 s clip
    for name in ("snn_c5_linear64", "snn_c5_random64"):
        g = H.load(name)
        T5 = 480_000
        f0 = float(np.mean(g["band"]))
        x = synthesize_clips(g["r_vec"], g["theta_vec"], FS, T5, rng.uniform(0.3, 2.8, args.extra_c5_clips),
                             snr_lin=np.full(args.extra_c5_clips, 10.0), sine_freq=f0, mode=0, seed=73, device=local)
        key = "c5_" + name.split("_")[-1]
        fp32_entry(key, g, x[:, :T], 1, fused=False, what="")
        par = res[key]["parity"]; cpu = res[key]["cpu_port"]
        fp32_entry(key, g, x, 0, fused=False,
                   what=f"configs[4]: {args.extra_c5_clips} x 10 s clips, 64-mic {name.split('_')[-1][:-2]} array, G=512")
        res[key]["parity"] = dict(par, note="first second of clip 0 against the oracle (the full 10 s clip is "
                                            "tests/test_gpu_parity.py::test_full_size_config5)")
        res[key]["cpu_port"] = dict(cpu, note="1 s of one 64-mic clip")
        one_ms, _ = _timed(torch, lambda: SnnEngineCache.run(g, x[:1], local))
        res[key]["one_clip_ms"] = one_ms
        del x
        if name == "snn_c5_linear64":
            # the same array as a Monte-Carlo batch: many one-second clips (unsegmented chains, tensor-core STHT / Gram)
            nb5 = 256
            xb = synthesize_clips(g["r_vec"], g["theta_vec"], FS, T, rng.uniform(0.3, 2.8, nb5), snr_lin=np.full(nb5, 10.0),
                                  sine_freq=f0, mode=0, seed=74, device=local)
            fp32_entry("c5_linear64_batch", g, xb, 0, fused=False,
                       what=f"{nb5} x 1 s clips on the 64-mic linear array of configs[4], G=512")
            del xb

    # design time (SURVEY 8f rank 1): SNNBeamformer.design_from_template on the G = 449 grid of configs[1] -- per-DoA front
    # end + neuron filter + covariance batched on the GPU (micloc_snn_gram), the 449 small eigen-problems on the host
    try:
        import contextlib
        import io
        from haghighatshoarmuir2024_b200.array_geometry import CenterCircularArray
        from haghighatshoarmuir2024_b200.snn_beamformer import SNNBeamformer
        d2, bands2 = load_workload()
        band = bands2[0]
        beamf = SNNBeamformer(CenterCircularArray(radius=4.5e-2, num_mic=NUM_MIC), float(d2["kernel_duration"]), band,
                              [float(d2["tau_0"])] * 2, bipolar_spikes=True, fs=FS, device=local)
        tt = np.arange(0, 0.25, 1 / FS)
        tmpl = (tt, np.sin(2 * np.pi * float(np.mean(band)) * tt))
        doa_list = np.linspace(-np.pi, np.pi, 449)
        with contextlib.redirect_stdout(io.StringIO()):
            beamf.design_from_template(tmpl, doa_list)
            t0 = time.perf_counter()
            bf = beamf.design_from_template(tmpl, doa_list)
            dt_design = time.perf_counter() - t0
        res["design_from_template"] = {
            "workload": "SNNBeamformer.design_from_template, 7-mic array, 0.25 s sine template, G=449 (micloc/snn_beamformer.py:82-211)",
            "seconds": dt_design, "doa_per_sec": 449 / dt_design, "bf_shape": list(bf.shape),
            "note": "front end + neuron filter + covariance of all DoAs in one batch on the GPU (staged kernels, float64 Gram); "
                    "the per-DoA SVD / constrained eigenvector stays on the host (numpy)"}
    except Exception as e:
        res["design_from_template"] = {"error": f"{type(e).__name__}: {e}"}

    # configs[2]: Xylo integer chain, bit-exact float64 front end + integer LIF network
    g = H.load("xylo_c3_bipolar")
    net = H.xylo_network(g)
    eng = H.xylo_engine(g, net, device=local)
    xs = torch.from_numpy(H.xylo_synth_clips(g, 16, T, seed=1)).to(f"cuda:{local}")
    Bx = args.extra_xylo_clips
    x = xs.repeat((Bx + 15) // 16, 1, 1)[:Bx].contiguous()
    x[16:] += 1e-3 * torch.randn_like(x[16:])                      # distinct clips; the first 16 stay the oracle's
    ms_exact, out = _timed(torch, lambda: eng.run(x, exact=True), n=2)           # audio in, counts + DoA out
    chk = eng.run(x[:16], exact=True, want_spikes_in=True)                       # the oracle's clips, with their input spikes
    out["spikes_in"] = chk["spikes_in"]
    spikes = eng.run(x, exact=True, want_spikes_in=True)["spikes_in"]
    ms_lif, _ = _timed(torch, lambda: eng.process(spikes, want_raster=False), n=2)
    del spikes
    ms_fast, outf = _timed(torch, lambda: eng.run(x, exact=False), n=2)
    n_cmp = 64
    t0 = time.perf_counter()
    ocfg = H.xylo_oracle_cfg(g, net)
    ref = O.xylo_run_batch(ocfg, x[:n_cmp].cpu().numpy(), FS, nthreads=min(cores, n_cmp))
    cpu_s = time.perf_counter() - t0
    ref["spikes_in"] = np.stack([O.xylo_encode(ocfg, xs[i].cpu().numpy())[0] for i in range(2)])
    v = ctypes.c_double()
    N_ = lib.micloc_fp32_peak(local, 2, ctypes.byref(v))
    fp64_peak = v.value if N_ == 0 else None               # DFMA TFLOP/s; DMUL + DADD pairs issue at the same rate
    M = x.shape[2]
    nb_ = len(g["bands"])
    ops = len(g["kernel"]) + nb_ * 2 * (2 * g["ba_b"].shape[1] - 1 + 2)   # un-fused f64 mul/add per mic-sample: STHT + band filters + cumsum
    front_ms = max(ms_exact - ms_lif, 1e-6)
    ach64 = Bx * T * M * ops / (front_ms * 1e-3) / 1e12
    res["c3_xylo"] = {
        "workload": "configs[2]: Xylo-quantised integer chain (int8 weights, bipolar RZCC, 449 hidden neurons, 28 inputs), "
                    "1 s chirp clips; exact = float64 front end in scipy's operation order + integer LIF",
        "clips": Bx, "exact_clips_per_sec": Bx / ms_exact * 1e3, "exact_ms": ms_exact,
        "lif_only_clips_per_sec": Bx / ms_lif * 1e3, "fp32_front_end_clips_per_sec": Bx / ms_fast * 1e3,
        "fp32_front_end_doa_agreement_with_exact": float((out["doa"] == outf["doa"]).float().mean()),
        "roofline_front_end": {"bound": "fp64 issue", "ops_per_mic_sample": ops, "achieved": ach64,
                               "peak": None if fp64_peak is None else fp64_peak / 2, "unit": "T f64 mul|add /s",
                               "frac": None if not fp64_peak else ach64 / (fp64_peak / 2),
                               "note": "front-end time = exact chain - LIF-only; peak = measured DFMA instruction rate "
                                       "(micloc_fp32_peak variant 2) counted one op per instruction: scipy's order "
                                       "forbids fusing the multiply with the add"},
        "parity": {"clips_compared": n_cmp,
                   "input_spikes_bit_exact": bool(np.array_equal(out["spikes_in"][:2].cpu().numpy(), ref["spikes_in"])),
                   "hidden_counts_bit_exact": bool(np.array_equal(out["counts"][:n_cmp].cpu().numpy(), ref["counts"])),
                   "doa_bit_exact": bool(np.array_equal(out["doa"][:n_cmp].cpu().numpy(), ref["doa"])),
                   "pinned": "front end: bit-identical to the reference's Demo.spike_encoding (tests/golden/xylo_*.npz); "
                             "integer network: oracle restatement of XyloSim, UNPINNED (rockpool absent)"},
        "cpu_port": {"clips_per_sec": n_cmp / cpu_s, "cores": min(cores, n_cmp)},
    }
    eng.close()
    return res


class SnnEngineCache:
    """One staged engine per golden case for the single-clip latency figure of config 5."""
    _e = {}

    @classmethod
    def run(cls, g, x, local):
        from haghighatshoarmuir2024_b200.engine import SnnEngine
        import helpers as H
        key = (id(g), x.shape[1])
        if key not in cls._e:
            cls._e[key] = SnnEngine(H.chain_spec(g, x.shape[1]), g["bf_mat"], device=local)
        return cls._e[key].run(x, want_spikes=True, want_power=True, fused=False)


def emit(line):
    """The contract is ONE JSON line on stdout: libraries (NCCL prints its version banner) write to fd 1 too, so
    fd 1 points at stderr for the whole run and the line goes to the original stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips-per-band", type=int, default=7104,
                    help="clips per band per step; 7104 = 12 x (148 SMs x 2 groups x 2 clips): the fused kernel hands clip pairs "
                         "to its persistent warp groups dynamically, a step should hold many pairs per group")
    ap.add_argument("--e2e-clips-per-band", type=int, default=1776, help="clips per band per step of the host-buffer (e2e) leg")
    ap.add_argument("--no-band-streams", dest="band_streams", action="store_false",
                    help="run the three band launches of a step back to back on one stream")
    ap.add_argument("--dtype", default="f32", choices=["f32", "i16"])
    ap.add_argument("--cpu-clips-per-band", type=int, default=0, help="CPU sample size per band (0 = auto)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs 1/3/4/5 section of the line")
    ap.add_argument("--extra-clips", type=int, default=1776, help="clips per extra config (1 s, 7 microphones)")
    ap.add_argument("--extra-xylo-clips", type=int, default=3552,
                    help="clips of the config-3 extra (3552 = 148 SMs x 24: one full wave of the exact front end's one-warp-per-clip kernel)")
    ap.add_argument("--extra-c5-clips", type=int, default=4, help="10 s 64-microphone clips of the config-5 extra")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
