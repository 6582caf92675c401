#!/usr/bin/env python
"""Benchmark of the one hot path: FullSubNet+ / FullSubNet inference on synthetic 16 kHz clips.

    python bench.py --gpus N --steps K --warmup W [--config 2|4|5]     # product arm (sm_100a kernels behind the C ABI)
    python bench.py --impl reference --gpus N --steps K ... [--config] # reference arm: the reference's own CPU PyTorch path

Metric (BASELINE.json): frames/sec and real-time factor.  Workloads (BASELINE.json configs, 1-based like BASELINE.md):
  --config 2 (default)  FullSubNet+ default config/inference.toml, 64 x 3 s clips per GPU per step (weak scaling; N = 8 is configs[2])
  --config 4            streaming: fullsubnet.Model + cumulative_laplace_norm, look_ahead 2, one 30 s clip frame by frame through the
                        step API, one frame per step (--steps 1876 = the whole clip); per-frame latency p50 / p99 (+ the offline
                        forwards of both models on the same clip)
  --config 5            large model: num_freqs 513 (n_fft 1024, hop 512), hidden 512, 3-layer LSTMs, 32 x 3 s clips

Configs 2 / 5, what one "step" is (identical at every N, so the driver's scaling efficiency compares like with like):
  value     the enhancement of one batch per GPU with the STFT-domain inputs resident in HBM, through the pipelined API
            (fsnplus_b200.inference.EnhancePipeline over fsn_model_submit): model forward -> decompress_cIRM x noisy spectrum
            -> torch.istft -> for N > 1 ONE NCCL all-gather of the enhanced waveforms.  Post-processing and the collective of
            batch i run on a side stream underneath the forward of batch i+1; everything is drained inside the timed region.
  e2e       the same loop with HOST buffers: pinned host spectra -> H2D (copy stream) -> ... -> D2H of this rank's enhanced
            waveforms into pinned host memory, every step.
  extras    forward_only (plain fsn_model_forward loop, the round-1 `value`), e2e_cabi (fsn_model_forward_host_async loop: mask to
            host, the round-1 `e2e`), cudnn_baseline (the reference model on the same B200 through stock PyTorch / cuDNN),
            cpu_baseline (+ .concurrent: as many B=1 workers as the host has cores for).
Prints ONE JSON line on rank 0.  ``--dump-outputs DIR`` then writes what the timed path (`value`) returned in its last step as
DIR/<name>.npy in float32 (configs 2 / 5: ``enhanced`` [N, samples], the waveforms of every rank; config 4: ``mask`` [B, 2, F], the
mask the last step returned), at most 64 MB in all; the inputs and the weights are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True                  # the benchmark leaves the tree as it found it (it may be read-only)
sys.path[:0] = [ROOT, os.path.join(ROOT, "fullsubnet-plus_b200")]

SR = 16000
DUMP_BYTES = 64 * 10 ** 6                       # --dump-outputs: budget of all files together


# ------------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------------
def plus_cfg(**over):
    """config/inference.toml:30-44 of the reference."""
    c = dict(sb_num_neighbors=15, fb_num_neighbors=0, num_freqs=257, look_ahead=2, sequence_model="LSTM",
             fb_output_activate_function="ReLU", sb_output_activate_function=False, channel_attention_model="TSSE",
             fb_model_hidden_size=512, sb_model_hidden_size=384, weight_init=False,
             norm_type="offline_laplace_norm", num_groups_in_drop_band=2, kersize=[3, 5, 10], subband_num=1)
    c.update(over)
    return c


default_cfg = plus_cfg          # name used by scripts/ and tests/dist_check.py


def fsn_cfg(**over):
    """fullsubnet.Model with the same hyper-parameters (reference fullsubnet.py:13-26)."""
    c = dict(sb_num_neighbors=15, fb_num_neighbors=0, num_freqs=257, look_ahead=2, sequence_model="LSTM",
             fb_output_activate_function="ReLU", sb_output_activate_function=False, fb_model_hidden_size=512,
             sb_model_hidden_size=384, weight_init=False, norm_type="offline_laplace_norm", num_groups_in_drop_band=2)
    c.update(over)
    return c


def workload(config, batch):
    if config == 2:
        return dict(id=2, kind="plus", cfg=plus_cfg(), L=2, B=batch or 64, nsamp=48000, n_fft=512, hop=256, T=188, clip_s=3.0,
                    name=f"FullSubNet+ default config/inference.toml, batch={batch or 64} synthetic 3 s 16 kHz clips per GPU (BASELINE configs[1])")
    if config == 5:
        return dict(id=5, kind="plus", cfg=plus_cfg(num_freqs=513, sb_model_hidden_size=512, fb_model_hidden_size=512), L=3, B=batch or 32,
                    nsamp=48000, n_fft=1024, hop=512, T=94, clip_s=3.0,
                    name=f"large FullSubNet+: num_freqs=513 (n_fft 1024, hop 512), hidden 512, 3-layer LSTMs, batch={batch or 32} synthetic 3 s clips "
                         "per GPU (BASELINE configs[4])")
    if config == 4:
        return dict(id=4, kind="fsn", cfg=fsn_cfg(norm_type="cumulative_laplace_norm"), L=2, B=batch or 1, nsamp=480000, n_fft=512, hop=256,
                    T=1876, clip_s=30.0,
                    name="streaming / causal: fullsubnet.Model + cumulative_laplace_norm, look_ahead=2, one 30 s synthetic clip frame by frame "
                         "(BASELINE configs[3])")
    raise SystemExit(f"unknown --config {config}")


def flops_per_clip(w):
    """Algorithmic FLOPs (SURVEY.md 8d).  Returns (sub-band LSTM + Linear, total)."""
    c, L, T_in = w["cfg"], w["L"], w["T"]
    F, Tp, H = c["num_freqs"], T_in + c["look_ahead"], c["sb_model_hidden_size"]
    nfb = 3 if w["kind"] == "plus" else 1
    I = (2 * c["sb_num_neighbors"] + 1) + nfb * (2 * c["fb_num_neighbors"] + 1)
    sb = Tp * F * (2 * 4 * H * (I + H) + (L - 1) * 2 * 4 * H * 2 * H + 2 * H * 2)
    if w["kind"] == "plus":
        tcn = 3 * Tp * (8 * (2 * 2 * F * 512 + 2 * 3 * 512) + 2 * F * F)
        ts = 3 * (2 * F * sum(c["kersize"]) * Tp + 4 * F * (F // 2))
        return sb, sb + tcn + ts
    Hf = c["fb_model_hidden_size"]
    fb = Tp * (2 * 4 * Hf * (F + Hf) + (L - 1) * 2 * 4 * Hf * 2 * Hf + 2 * Hf * F)
    return sb, sb + fb


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons, pw = [], 0, set(), []
        for ts, line in self.rows:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9 or not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[1])); mx = max(mx, float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return None
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm),
                "power_w_median": statistics.median(pw) if pw else None}


# ------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own CPU PyTorch path (oracle/_ref = verbatim copy of the reference, else the torch port)
# ------------------------------------------------------------------------------------------------------------------
def make_cpu_model(params, w):
    """Returns (callable forward(mag, real, imag) for ONE clip, kind).  kind = "reference": the unmodified reference class from
    oracle/_ref (or /root/reference); "port": oracle/torch_port.py (same ATen op sequence) when the reference is absent or the
    workload uses the additive num_layers knob the reference constructor does not have."""
    from oracle import ref_loader
    if ref_loader.available() and w["L"] == 2:
        m = ref_loader.ReferenceCpu(params, w["cfg"], w["kind"])
        return m.forward, "reference"
    from oracle.torch_port import TorchPort
    m = TorchPort(params, w["cfg"], w["kind"], num_layers=w["L"])
    return m.forward, "port"


def cpu_time_clips(fwd, spec, n, start=0):
    mag, real, imag = spec
    out = []
    for i in range(n):
        j = (start + i) % mag.shape[0]
        t0 = time.perf_counter()
        fwd(mag[j:j + 1], real[j:j + 1] if real is not None else None, imag[j:j + 1] if imag is not None else None)
        out.append(time.perf_counter() - t0)
    return out


def thread_sweep(fwd, spec):
    """Best intra-op thread count for B=1 calls (torch's default of one thread per core is ~80x slower than 16 threads on the
    128-core GPU hosts for these small GEMMs; the baseline is reported at its best setting, not its default)."""
    import torch
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (1, 4, 8, 16, 32, 64, ncpu) if c <= ncpu})
    sweep, best, threads = {}, None, cands[0]
    for c in cands:
        torch.set_num_threads(c)
        cpu_time_clips(fwd, spec, 1)
        t = min(cpu_time_clips(fwd, spec, 2))
        sweep[c] = round(t, 3)
        if best is None or t < best:
            best, threads = t, c
        elif t > 1.8 * best:
            break
    torch.set_num_threads(threads)
    return threads, sweep


def _cpu_worker(conn, params, w, spec, threads):
    """One concurrent B=1 worker (spawned process): build the CPU model, then run `n` clips per request."""
    import torch
    torch.set_num_threads(threads)
    sys.path[:0] = [ROOT]
    fwd, _ = make_cpu_model(params, w)
    cpu_time_clips(fwd, spec, 1)
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg is None:
            break
        t0 = time.perf_counter()
        cpu_time_clips(fwd, spec, msg)
        conn.send(time.perf_counter() - t0)


class CpuWorkers:
    """`nworkers` processes x `threads` intra-op threads, each enhancing its own clips one per call: the throughput-fair CPU
    figure (the reference inferencer is single-process B=1; a user with a 128-core host would run several)."""

    def __init__(self, params, w, spec, threads, nworkers):
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        self.conns, self.procs = [], []
        for _ in range(nworkers):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(b, params, w, spec, threads), daemon=True)
            p.start()
            self.conns.append(a); self.procs.append(p)
        for c in self.conns:
            assert c.recv() == "ready"

    def step(self, clips_per_worker):
        t0 = time.perf_counter()
        for c in self.conns:
            c.send(clips_per_worker)
        for c in self.conns:
            c.recv()
        return time.perf_counter() - t0

    def close(self):
        for c in self.conns:
            c.send(None)
        for p in self.procs:
            p.join(timeout=10)


def host_spec(w, n, seed=1000):
    """n clips of the workload -> CPU spectra ([n,1,F,T] mag/real/imag float32)."""
    from fsnplus_b200.synth import synth_clips
    from fsnplus_b200 import inference as inf
    nsamp = 48000 if w["id"] == 4 else w["nsamp"]              # the CPU sample of the streaming config is a 3 s clip (bounded)
    X = inf.stft(synth_clips(n, nsamp, SR, seed=seed), w["n_fft"], w["hop"], w["n_fft"])
    if w["kind"] == "plus":
        return (X.abs().unsqueeze(1).contiguous(), X.real.unsqueeze(1).contiguous(), X.imag.unsqueeze(1).contiguous())
    return (X.abs().unsqueeze(1).contiguous(), None, None)


def reference_arm(args, w, state):
    import torch
    params = {k: v.detach().cpu().numpy() for k, v in state.items()}
    n = args.ref_clips
    spec = host_spec(w, max(n, 2))
    frames = spec[0].shape[-1]
    clip_s = 3.0 if w["id"] == 4 else w["clip_s"]
    fwd, kind = make_cpu_model(params, w)
    threads, sweep = thread_sweep(fwd, spec)
    single = statistics.median(cpu_time_clips(fwd, spec, max(3, n)))
    ncpu = os.cpu_count() or 1
    nworkers = max(1, min(ncpu // threads, 16))
    pool = CpuWorkers(params, w, spec, threads, nworkers)
    K, W = args.steps, args.warmup
    times = []
    for s in range(W + K):
        t = pool.step(n)
        if s >= W:
            times.append(t)
    pool.close()
    per_step = statistics.median(times)
    fps_conc = nworkers * n * frames / per_step
    fps_single = frames / single
    # the arm's value is the reference CPU path at its BEST use of the host: several concurrent B=1 workers or one process,
    # whichever is faster (on the 128-core GPU hosts the workers are memory-bound and one 16-thread process wins)
    use_conc = fps_conc >= fps_single
    fps = fps_conc if use_conc else fps_single
    step_ms = per_step * 1e3 if use_conc else single * n * 1e3
    line = {
        "impl": "reference", "metric": "frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "rtf": (per_step / (nworkers * n * clip_s)) if use_conc else single / clip_s,
        "config": {"workload": w["name"]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": nworkers * threads if use_conc else threads, "kind": kind,
                         "sample": (f"{nworkers} concurrent worker processes x {threads} threads, {n} clips per worker per step x {K} steps" if use_conc else
                                    f"one process x {threads} threads (faster than {nworkers} concurrent workers on this host), {max(3, n)} clips")
                                   + f", one 3 s clip per call (the reference inference batch size), model forward only, torch {torch.__version__} CPU fp32"
                                   + (" (the reference cannot stream: offline forward of 3 s clips)" if w["id"] == 4 else ""),
                         "host_cores": ncpu, "thread_sweep_s_per_clip": sweep,
                         "single_process": {"value": fps_single, "unit": "frames/s", "cores": threads, "rtf": single / clip_s},
                         "concurrent": {"value": fps_conc, "unit": "frames/s", "workers": nworkers, "threads_per_worker": threads, "ms_per_step": per_step * 1e3}},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------
# product arm, configs 2 / 5
# ------------------------------------------------------------------------------------------------------------------
def product_batched(args, w, model, state, rank, local_rank, world, make_model, outputs):
    import torch
    import torch.distributed as dist
    from fsnplus_b200.synth import synth_clips
    from fsnplus_b200 import inference as inf
    dev = torch.device("cuda", local_rank)
    cfg, B, K, W, T, F = w["cfg"], w["B"], args.steps, max(args.warmup, 3), w["T"], w["cfg"]["num_freqs"]
    stft_args = (w["n_fft"], w["hop"], w["n_fft"])

    # inputs: NSETS distinct batches rotated so consecutive steps never reuse L2-resident inputs
    NSETS = 4
    clips = synth_clips(NSETS * B, w["nsamp"], SR, seed=1000 + 7919 * rank).to(dev)
    X = inf.stft(clips, *stft_args).reshape(NSETS, B, F, T)
    assert X.shape[-1] == T
    Xs = [X[i].contiguous() for i in range(NSETS)]
    mags = [x.abs().unsqueeze(1).contiguous() for x in Xs]
    reals = [x.real.unsqueeze(1).contiguous() for x in Xs]
    imags = [x.imag.unsqueeze(1).contiguous() for x in Xs]
    in_bytes = 3 * B * F * T * 4
    wav_bytes = B * w["nsamp"] * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(body, steps, warm, drain=None):
        """`body(i)` enqueues step i; `drain()` (inside the timed region) completes everything enqueued."""
        with torch.no_grad():
            for i in range(warm):
                body(i)
            if drain:
                drain()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.time()
            e0.record()
            for i in range(steps):
                body(warm + i)
            timed.host_ms = (time.time() - t0) * 1e3 / steps          # host time to ENQUEUE one step (before the drain)
            if drain:
                drain()
            e1.record()
            barrier()
            t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item() / steps, t0, t1

    # ---- forward_only: the plain forward loop (round-1 `value`), also the un-overlapped kernel timings --------------------
    ms_fwd, _, _ = timed(lambda i: model(mags[i % NSETS], reals[i % NSETS], imags[i % NSETS]), K, W)
    lstm_ms_plain = [x for x in model.lstm_ms_history(min(K, 32)) if x > 0]
    launches_fwd = model.last_launch_count()
    lstm_impl = model.last_lstm_impl()

    # ---- value: pipelined enhancement, inputs resident in HBM, collective inside the timed region -------------------------
    pipe = inf.EnhancePipeline(model, w["nsamp"], *stft_args, gather=True, to_host=False, keep_results=False)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    ms_step, t0, t1 = timed(lambda i: pipe.push(Xs[i % NSETS]), K, max(W, pipe.NSLOT + 1), drain=pipe.flush)   # warm-up fills every ring slot (allocations)
    host_ms = timed.host_ms
    outputs["enhanced"] = pipe.last.cpu().numpy()                 # the last timed step's waveforms (all ranks' when gathered)
    clocks = sampler.stop(t0, t1) if sampler else None
    lstm_ms = [x for x in model.lstm_ms_history(min(K, 32)) if x > 0]
    fps = world * B * T / (ms_step * 1e-3)

    # ---- experiment: front end of batch i+1 CONCURRENT with the sub-band LSTM of batch i (FSN_FRONT_OVERLAP=1, read at model creation) ------
    overlap = None
    if world == 1 and not args.no_overlap_experiment:
        os.environ["FSN_FRONT_OVERLAP"] = "1"
        m2 = make_model().to(dev)
        m2.load_state_dict(state)
        pipe2 = inf.EnhancePipeline(m2, w["nsamp"], *stft_args, gather=False, to_host=False, keep_results=False)
        ms2, _, _ = timed(lambda i: pipe2.push(Xs[i % NSETS]), K, max(W, pipe2.NSLOT + 1), drain=pipe2.flush)
        del os.environ["FSN_FRONT_OVERLAP"]
        k2 = [x for x in m2.lstm_ms_history(min(K, 32)) if x > 0]
        overlap = {"ms_per_step": ms2, "lstm_kernel_ms": statistics.mean(k2) if k2 else None,
                   "timeline_ms": {"columns": ["front_start", "front_end", "lstm_start", "lstm_end"], "last_steps": [[round(x, 3) for x in r] for r in m2.timeline(6)]},
                   "note": "same loop with the front end of batch i+1 on a second stream / workspace lane while the LSTM of batch i runs on its 130 SMs: the front "
                           "end lies inside the LSTM interval, and the LSTM kernel slows down by about the front end's stand-alone time (power-capped) -> off by default"}
        del pipe2, m2

    # ---- e2e: same loop, pinned host spectra in, this rank's enhanced waveforms out to pinned host memory --------------------
    pin = lambda x: x.cpu().pin_memory()
    hosts = [(pin(mags[i]), pin(reals[i]), pin(imags[i])) for i in range(NSETS)]
    pipe_h = inf.EnhancePipeline(model, w["nsamp"], *stft_args, gather=True, to_host=True, keep_results=False)
    ms_e2e, _, _ = timed(lambda i: pipe_h.push(host=hosts[i % NSETS]), K, max(W, pipe_h.NSLOT + 1), drain=pipe_h.flush)   # warm-up fills every ring slot
    fps_e2e = world * B * T / (ms_e2e * 1e-3)

    # ---- e2e_cabi: the C ABI's own host-buffer entry point (mask to host; the round-1 `e2e`) ------------------------------------
    houts = [torch.empty((B, 2, F, T), dtype=torch.float32).pin_memory() for _ in range(2)]

    def cabi_step(i):
        model.forward_host(*hosts[i % NSETS], out=houts[i % 2], device=dev, pipelined=True)
    ms_cabi, _, _ = timed(cabi_step, K, 3, drain=model.sync_host)

    if rank != 0:
        return None

    sb_flops, tot_flops = flops_per_clip(w)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        pk = json.load(open(peaks_path))
        peak, peak_burst, peak_src = pk["bf16_tflops_sustained"], pk["bf16_tflops"], "measured (MEASURED_PEAKS.json, sustained)"
    else:
        peak, peak_burst, peak_src = 1400.0, 1590.0, "fallback (B200_PROFILING.md)"
    traffic = None                                    # dram read+write bytes per launch from the committed ncu --set full capture
    tpath = os.path.join(ROOT, "profiles", "lstm_traffic.json")
    if os.path.exists(tpath) and lstm_impl == "tcgen05" and B == 64 and w["id"] == 2:
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    k_ms = statistics.mean(lstm_ms) if lstm_ms else float("nan")
    k_ms_plain = statistics.mean(lstm_ms_plain) if lstm_ms_plain else float("nan")
    achieved = B * sb_flops / (k_ms * 1e-3) / 1e12
    roofline = {"bound": "tensor", "kernel": f"sub-band LSTM ({lstm_impl}" + (", layer-wise: all layers incl. input-projection GEMMs" if w["L"] != 2 or cfg["sb_model_hidden_size"] > 384 else "") + ")",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "frac_of_burst_peak": achieved / peak_burst, "peak_source": peak_src,
                "kernel_ms": k_ms, "kernel_ms_without_overlap": k_ms_plain, "kernel_share_of_step": k_ms / ms_step, "traffic": traffic,
                "algorithmic_flops_per_launch": B * sb_flops,
                "timing": "CUDA events around the kernel on the stream it is launched on (inside the library), mean over the timed steps of `value` "
                          "(the iSTFT of the previous batch runs on a side stream underneath it)"}
    line = {
        "metric": "frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "rtf": ms_step * 1e-3 / (B * w["clip_s"]),
        "config": {"workload": w["name"], "config_id": w["id"], "clips_per_gpu": B, "frames_per_clip": T, "lstm_impl": lstm_impl,
                   "gate_math": "ex2+rcp" if args.accurate_math else "tanh.approx (default)", "weights": "random init (torch default, seed 0)",
                   "step": "model forward -> decompress_cIRM x spectrum -> torch.istft" + (" -> ONE NCCL all_gather_into_tensor of the enhanced waveforms "
                           f"({world} ranks, {world * wav_bytes / 1e6:.0f} MB gathered, side stream, inside the timed region)" if world > 1 else "")
                           + "; pipelined (fsn_model_submit_enhance): the cIRM post-processing is fused into the LSTM epilogue, iSTFT"
                           + (" and the collective" if world > 1 else "") + " of batch i-1 run on a side stream under the forward of batch i",
                   "l2": f"inputs rotated over {NSETS} batches ({NSETS * in_bytes / 1e6:.0f} MB > L2); per-step intermediates exceed L2"},
        "model_tflops": world * B * tot_flops / (ms_step * 1e-3) / 1e12,
        "host_enqueue_ms_per_step": host_ms,
        "roofline": roofline,
        "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": ms_e2e, "rtf": ms_e2e * 1e-3 / (B * w["clip_s"]),
                "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": wav_bytes,
                "path": "fsnplus_b200.inference.EnhancePipeline: pinned host spectra -> H2D (copy stream) -> fsn_model_submit -> cIRM -> istft"
                        + (" -> NCCL all-gather" if world > 1 else "") + " -> D2H of this rank's enhanced waveforms (pinned), all drained inside the timed region"},
        "forward_only": {"value": world * B * T / (ms_fwd * 1e-3), "unit": "frames/s", "ms_per_step": ms_fwd, "launches_per_step": launches_fwd,
                         "path": "fsn_model_forward in a loop on one stream (no cross-batch overlap; the round-1 `value`)"},
        "e2e_cabi": {"value": world * B * T / (ms_cabi * 1e-3), "unit": "frames/s", "ms_per_step": ms_cabi,
                     "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 2 * B * F * T * 4,
                     "path": "fsn_model_forward_host_async (C ABI, pinned host buffers, mask to host; the round-1 `e2e`)"},
        "gpu_launches": launches_fwd * K,                      # this library's kernels in the timed region of `value` (the cIRM pass is fused into the LSTM epilogue)
        "clocks": clocks,
        "front_overlap_experiment": overlap,
    }
    return line


# ------------------------------------------------------------------------------------------------------------------
# product arm, config 4 (streaming)
# ------------------------------------------------------------------------------------------------------------------
def product_streaming(args, w, model, state, rank, local_rank, world, outputs):
    import numpy as np
    import torch
    from fsnplus_b200.synth import synth_clips
    from fsnplus_b200 import inference as inf
    from fsnplus_b200.streaming import StreamingFullSubNet
    from fsnplus_b200.model import FullSubNet_Plus
    dev = torch.device("cuda", local_rank)
    B, F = w["B"], w["cfg"]["num_freqs"]
    clip = synth_clips(B, w["nsamp"], SR, seed=77 + rank).to(dev)
    X = inf.stft(clip)
    mag = X.abs().contiguous()                                    # [B, 257, 1876]
    T = mag.shape[-1]
    frames = [mag[:, :, t].contiguous() for t in range(T)]
    hframes = [f.cpu().pin_memory() for f in frames]
    K = args.steps
    if K > T:
        raise SystemExit(f"--steps {K}: the {w['clip_s']:.0f} s clip has {T} frames (one frame per step)")

    def run(host):
        st = StreamingFullSubNet(model, batch_size=B, device=dev)
        for t in range(20):
            st.step(frames[t])
        torch.cuda.synchronize()
        st.close()
        st = StreamingFullSubNet(model, batch_size=B, device=dev)
        hout = torch.empty((B, 2, F), dtype=torch.float32).pin_memory()
        stage = torch.empty((B, F), dtype=torch.float32, device=dev)
        lat, dev_ms = [], []
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for t in range(K):
            t0 = time.perf_counter()
            if host:
                stage.copy_(hframes[t], non_blocking=True)
                y = st.step(stage)
                if y is not None:
                    hout.copy_(y, non_blocking=True)
            else:
                evs[t][0].record()
                y = st.step(frames[t])
                evs[t][1].record()
            torch.cuda.synchronize()                              # a real-time caller needs the mask before the next hop
            lat.append((time.perf_counter() - t0) * 1e3)
        if not host:
            dev_ms = [a.elapsed_time(b) for a, b in evs]
            outputs["mask"] = y.cpu().numpy() if y is not None else None
        st.close()
        return np.array(lat), np.array(dev_ms)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.3)
    t0 = time.time()
    lat, dev_ms = run(False)
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if sampler else None
    lat_h, _ = run(True)

    # offline forwards on the same 30 s clip (FullSubNet+ cannot stream: TSSE pools over all time, SURVEY.md 0.5)
    def offline(m, *ins):
        with torch.no_grad():
            for _ in range(2):
                m(*ins)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                m(*ins)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 3
    off_fsn = offline(model, mag.unsqueeze(1))
    torch.manual_seed(0)
    plus = FullSubNet_Plus(**plus_cfg()).eval().to(dev)
    off_plus = offline(plus, mag.unsqueeze(1), X.real.unsqueeze(1).contiguous(), X.imag.unsqueeze(1).contiguous())
    if rank != 0:
        return None
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm = json.load(open(peaks_path))["hbm_gbs"] if os.path.exists(peaks_path) else 6500.0
    # algorithmic bytes per frame: every weight once (sub-band LSTM fp16 images, full-band LSTM fp32 parameters) -- activations are negligible
    c = w["cfg"]
    Hs, Hf, I = c["sb_model_hidden_size"], c["fb_model_hidden_size"], 2 * c["sb_num_neighbors"] + 2
    wbytes = 2 * (4 * Hs * (64 + Hs) + 4 * Hs * 2 * Hs) + 4 * (4 * Hf * (F + Hf) + 4 * Hf * 2 * Hf + F * Hf)
    mean_dev = float(dev_ms.mean())
    pct = lambda a, q: float(np.percentile(a, q))
    line = {
        "metric": "frames_per_sec", "value": B * 1e3 / float(lat.mean()), "unit": "frames/s", "n_gpus": world, "steps": int(K), "warmup": 20,
        "ms_per_step": float(lat.mean()), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "rtf": float(lat.mean()) / 16.0,
        "latency_ms": {"p50": pct(lat, 50), "p99": pct(lat, 99), "mean": float(lat.mean()), "max": float(lat.max()),
                       "device_p50": pct(dev_ms, 50), "device_p99": pct(dev_ms, 99), "hop_ms": 16.0, "algorithmic_latency_ms": 48.0,
                       "definition": "host wall clock per frame: enqueue of fsn_stream_step + synchronize (device_*: CUDA events around the step)"},
        "config": {"workload": w["name"], "config_id": 4, "streams": B, "frames": int(T), "step": "one fsn_stream_step (frame n in, mask of frame n-2 out), synchronised"},
        "roofline": {"bound": "hbm", "kernel": "streaming step (weight-stationary full-band LSTM step + generic sub-band step, launch-latency-bound)",
                     "achieved": wbytes / (mean_dev * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s", "frac": wbytes / (mean_dev * 1e-3) / 1e9 / hbm,
                     "traffic": None, "algorithmic_bytes_per_frame": wbytes, "kernel_ms": mean_dev},
        "e2e": {"value": B * 1e3 / float(lat_h.mean()), "unit": "frames/s", "ms_per_step": float(lat_h.mean()),
                "latency_ms": {"p50": pct(lat_h, 50), "p99": pct(lat_h, 99)},
                "h2d_bytes_per_step": B * F * 4, "d2h_bytes_per_step": B * 2 * F * 4,
                "path": "pinned host frame -> H2D -> fsn_stream_step -> D2H of the mask frame -> synchronize, every frame"},
        "offline_30s": {"fullsubnet_model_ms": off_fsn, "fullsubnet_plus_ms": off_plus, "rtf_model": off_fsn / 30e3, "rtf_plus": off_plus / 30e3},
        "gpu_launches": 6 * int(K),
        "clocks": clocks,
    }
    return line


# ------------------------------------------------------------------------------------------------------------------
# secondary baselines (N = 1, rank 0)
# ------------------------------------------------------------------------------------------------------------------
def cudnn_baseline(w, state, dev):
    """The reference model on the SAME B200 through stock PyTorch / cuDNN (SURVEY.md 8d "secondary baseline"): (a) the unmodified
    reference class, one clip per call, fp32, as its inferencer issues it (inferencer.py:149-151) but with a real synchronize;
    (b) the torch port (same ATen ops, per-sample semantics at any batch size) at the full batch, fp32 and fp16 autocast."""
    import torch
    from oracle import ref_loader
    from oracle.torch_port import TorchPort
    params = {k: v.detach().cpu().numpy() for k, v in state.items()}
    spec = [x.to(dev) if x is not None else None for x in host_spec(w, w["B"])]
    frames, out = spec[0].shape[-1], {}

    def ev_time(fn, reps):
        fn(); fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    with torch.no_grad():
        if ref_loader.available() and w["L"] == 2:
            ref = ref_loader.ReferenceCpu(params, w["cfg"], w["kind"])
            ref.model.to(dev)
            n = min(8, w["B"])
            ms = ev_time(lambda: [ref.forward(*(x[i:i + 1] if x is not None else None for x in spec)) for i in range(n)], 2) / n
            out["reference_b1_fp32"] = {"ms_per_clip": ms, "value": frames / (ms * 1e-3), "unit": "frames/s",
                                        "path": "unmodified reference class (oracle/_ref) .to(cuda), one clip per call, cuDNN LSTM"}
        port = TorchPort(params, w["cfg"], w["kind"], num_layers=w["L"])
        port.p = {k: v.to(dev) for k, v in port.p.items()}
        for m in port.lstm.values():
            m.to(dev)
        try:
            ms = ev_time(lambda: port.forward(*spec), 3)
            out["port_batched_fp32"] = {"ms_per_step": ms, "value": w["B"] * frames / (ms * 1e-3), "unit": "frames/s", "batch": w["B"],
                                        "path": "torch port (same ATen ops) at the full batch, cuDNN LSTM over B*F sequences"}
            with torch.autocast("cuda", dtype=torch.float16):
                ms = ev_time(lambda: port.forward(*spec), 3)
            out["port_batched_fp16_autocast"] = {"ms_per_step": ms, "value": w["B"] * frames / (ms * 1e-3), "unit": "frames/s", "batch": w["B"]}
        except Exception as e:                                      # e.g. out of memory on the unfold + cuDNN workspace
            out["port_batched_error"] = str(e)[:200]
    return out


def cpu_baseline(args, w, state):
    import torch
    params = {k: v.detach().cpu().numpy() for k, v in state.items()}
    n = args.cpu_baseline_clips
    spec = host_spec(w, n)
    frames = spec[0].shape[-1]
    clip_s = 3.0 if w["id"] == 4 else w["clip_s"]
    fwd, kind = make_cpu_model(params, w)
    threads, sweep = thread_sweep(fwd, spec)
    cpu_time_clips(fwd, spec, 1)
    times = cpu_time_clips(fwd, spec, n)
    med = statistics.median(times)
    ncpu = os.cpu_count() or 1
    out = {"value": frames / med, "unit": "frames/s", "cores": threads, "kind": kind, "rtf": med / clip_s,
           "sample": f"{n} clips of the workload, one 3 s clip per call (reference inference batch size), model forward only, torch {torch.__version__} "
                     f"CPU fp32, median of {n} after 1 warm-up" + (" (the reference cannot stream: offline forward of 3 s clips)" if w["id"] == 4 else ""),
           "host_cores": ncpu, "thread_sweep_s_per_clip": sweep}
    nworkers = max(1, min(ncpu // threads, 16))
    if nworkers > 1:
        pool = CpuWorkers(params, w, spec, threads, nworkers)
        pool.step(1)
        t = pool.step(3)
        pool.close()
        out["concurrent"] = {"value": nworkers * 3 * frames / t, "unit": "frames/s", "cores": nworkers * threads, "workers": nworkers,
                             "threads_per_worker": threads, "sample": "3 clips per worker, all workers at once (throughput-fair figure)"}
    return out


def dump_outputs(dirname, arrays):
    """Write each array as dirname/<name>.npy in float32.  Beyond DUMP_BYTES in all, every array keeps a fixed, seeded sample of
    its rows (first axis, in order) in proportion to its size; the same shapes always give the same sample."""
    import numpy as np
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items() if v is not None}
    if not arrays:
        raise SystemExit("--dump-outputs: the timed path returned nothing in its last step")
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            keep = max(1, DUMP_BYTES * a.shape[0] // total)
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(dirname, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 4, 5], help="BASELINE config (1-based): 2 = batch 64 default model, 4 = streaming, 5 = large model")
    ap.add_argument("--batch", type=int, default=0, help="clips per GPU per step (default: the config's)")
    ap.add_argument("--lstm-impl", default="auto", choices=["auto", "mma", "tcgen05"])
    ap.add_argument("--accurate-math", action="store_true", help="ex2/rcp gate math instead of the default tanh.approx path")
    ap.add_argument("--ref-clips", type=int, default=2, help="reference arm: clips per worker per step (bounded sample)")
    ap.add_argument("--cpu-baseline-clips", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cudnn-baseline", action="store_true")
    ap.add_argument("--no-overlap-experiment", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy (float32, <= 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")

    import torch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    w = workload(args.config, args.batch)

    from fsnplus_b200.model import FullSubNet_Plus, Model
    torch.manual_seed(0)
    extra = dict(lstm_impl=args.lstm_impl, fast_math=not args.accurate_math, num_layers=w["L"])
    make_model = lambda: (FullSubNet_Plus if w["kind"] == "plus" else Model)(**w["cfg"], **extra).eval()
    model = make_model()                                                                              # random init, seed 0
    state = model.state_dict()

    if args.impl == "reference":
        if rank == 0:
            reference_arm(args, w, state)
        return

    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a B200: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = model.to(dev)
    outputs = {}
    if w["id"] == 4:
        line = product_streaming(args, w, model, state, rank, local_rank, world, outputs)
    else:
        line = product_batched(args, w, model, state, rank, local_rank, world, make_model, outputs)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    if rank == 0:
        if world == 1 and not args.no_cudnn_baseline:
            try:
                line["cudnn_baseline"] = cudnn_baseline(w, state, dev)
            except Exception as e:
                line["cudnn_baseline"] = {"error": str(e)[:300]}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, w, state)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
