#!/usr/bin/env python
"""bench.py -- mel frames/sec of the Tacotron hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--mode infer] [--dump-outputs DIR]

A "step" is one pass of the hot path over one synthetic batch of BASELINE config 2:
B=32 utterances, char length 128, 200 decoder steps, r=5  (32 000 mel frames), free-running
inference forward (Tacotron.inference(train=False): encoder CBHG -> persistent attention decoder
-> post-processing CBHG -> linear-spectrogram dense).

Our arm: device-resident inputs, CUDA-event timing per step, L2 flushed between steps, max over
ranks; plus `e2e` (host pinned inputs -> H2D -> public API -> D2H of output + alignments),
`roofline` for the dominant kernel and `cpu_baseline` (the CPU oracle on the host cores).
--impl reference: the reference's CPU path stand-in (the PyTorch-CPU oracle port; TensorFlow 1.2
cannot be installed here) on the same config, all host threads.
N > 1: inference shards by utterance with no exchange -> N independent replicas (weak scaling).
--dump-outputs DIR: after the timed steps, rank 0 writes what its last timed step returned as DIR/<name>.npy (float32,
see dump_outputs); the inputs and weights are seeded, so two builds can be compared output for output.
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

B, TX, T, R = 32, 128, 200, 5
FRAMES = B * T * R
# forward FLOP (2*MAC), true unpadded contraction sizes, SURVEY.md section 8d / BASELINE.md section 3
FWD_GFLOP = 168.05
DECODER_GFLOP = 22.649 + 0.537          # decoder loop + attention memory layer (per launch at C2)
METRIC = "mel frames/sec at batch 32 r=5; decoder-step p50 latency"
WORKLOAD = "C2 synthetic: B=32, char 128, 200 decoder steps, r=5, inference forward (free-running)"


def config_dict(world, **extra):
    """the `config` object of the JSON line -- IDENTICAL (keys and values) in our arm and in the reference arm for the
    same N; what differs between the arms (precision mode, CUDA graphs) is reported under `run`"""
    c = {"workload": WORKLOAD, "frames_per_step": FRAMES, "batch": B, "char_len": TX, "decoder_steps": T, "r": R,
         "l2": "GPU arm: 256 MB flush write between timed steps; CPU reference arm: not applicable",
         "parallelism": f"replicas x{world}, no collective on the data path (the CPU reference arm runs on rank 0 only)"}
    c.update(extra)
    return c


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    FIELDS = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_step(params, inp, cfg):
    from oracle import tacotron_oracle as O
    import torch
    with torch.no_grad():
        return O.inference(params, inp, cfg, train=False)


CPU_THREADS_DEFAULT = 16
_cpu_threads = None            # chosen once per process (see pick_cpu_threads)


def _oracle_setup():
    import torch
    from oracle import tacotron_oracle as O
    cfg = O.OracleConfig(r=R, max_decode_iter=T)
    params = O.init_params(cfg, seed=1)
    inp = O.synthetic_inputs(cfg, B, TX, T, seed=0, with_targets=False)
    return cfg, params, inp


def shard_worker(threads, nshards, steps, warmup):
    """child process of time_cpu_oracle_sharded: the oracle forward on B / nshards utterances of the C2 batch with `threads`
    threads.  Warm-up, print "ready", wait for a line on stdin (the parent releases all shards together), `steps` timed
    forwards, print the elapsed seconds."""
    import torch
    from oracle import tacotron_oracle as O
    torch.set_num_threads(threads)
    cfg = O.OracleConfig(r=R, max_decode_iter=T)
    params = O.init_params(cfg, seed=1)
    inp = O.synthetic_inputs(cfg, B // nshards, TX, T, seed=0, with_targets=False)
    for _ in range(max(1, warmup)):
        cpu_oracle_step(params, inp, cfg)
    print("ready", flush=True)
    sys.stdin.readline()
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_oracle_step(params, inp, cfg)
    print(json.dumps({"sec": time.perf_counter() - t0}), flush=True)


def time_cpu_oracle_sharded(steps, warmup, nshards, threads, timeout=240):
    """The C2 batch split over `nshards` processes x `threads` threads (utterances are independent in inference: batch norm
    uses moving statistics, attention is per utterance).  One PyTorch-CPU process does not scale past ~16 threads on this
    workload (~3000 small ops per forward); sharding the batch is how the port uses ALL host cores.  Returns seconds per
    step = slowest shard's time for `steps` forwards / steps, or None when a shard fails."""
    procs = []
    try:
        for _ in range(nshards):
            procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), "--impl", "reference-shard", "--threads", str(threads),
                                           "--nshards", str(nshards), "--steps", str(steps), "--warmup", str(warmup)],
                                          stdin=subprocess.PIPE, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, cwd=ROOT))
        deadline = time.time() + timeout
        for pr in procs:                                    # every shard has warmed up
            line = pr.stdout.readline()
            if line.strip() != "ready" or time.time() > deadline:
                raise RuntimeError("shard did not get ready")
        for pr in procs:
            pr.stdin.write("go\n"); pr.stdin.flush()
        secs = []
        for pr in procs:
            out = pr.stdout.readline()
            secs.append(json.loads(out)["sec"])
        return max(secs) / steps
    except Exception:
        return None
    finally:
        for pr in procs:
            try:
                pr.kill()
            except Exception:
                pass


def probe_worker(threads):
    """child process of pick_cpu_threads: one warm-up + one timed C2 forward of the oracle at `threads` threads"""
    import torch
    torch.set_num_threads(threads)
    cfg, params, inp = _oracle_setup()
    cpu_oracle_step(params, inp, cfg)
    t0 = time.perf_counter()
    cpu_oracle_step(params, inp, cfg)
    print(json.dumps({"threads": threads, "sec": time.perf_counter() - t0}), flush=True)


def pick_cpu_threads(probe):
    """Thread count for the CPU arm.  The oracle is ~3000 small ops per forward and more threads are often SLOWER on
    this pool's hosts (round 1: 16 threads 37 K frames/s, 64 threads 3.9 K).  With `probe` (the --impl reference arm)
    16 / 32 / 64 threads are each tried once in a CHILD process (re-sizing the OpenMP pool inside one process cost
    minutes on the 64-core box) and the fastest is kept; otherwise 16."""
    global _cpu_threads
    if _cpu_threads is not None:
        return _cpu_threads
    ncpu = os.cpu_count() or 1
    best, tried = min(CPU_THREADS_DEFAULT, ncpu), {}
    if probe:
        best_sec = None
        for th in (16, 32, 64):
            if th > ncpu:
                continue
            try:
                out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-probe", "--threads", str(th)],
                                     capture_output=True, text=True, timeout=150, cwd=ROOT)
                sec = json.loads(out.stdout.strip().splitlines()[-1])["sec"]
                tried[th] = sec
                if best_sec is None or sec < best_sec:
                    best, best_sec = th, sec
            except Exception as ex:                         # a probe that fails or times out is simply not chosen
                tried[th] = f"failed: {type(ex).__name__}"
    _cpu_threads = (best, tried, ncpu)
    return _cpu_threads


def time_cpu_oracle(iters, warmup=1, probe=False):
    """The reference's CPU path stand-in: PyTorch-CPU fp32 oracle on the host cores, C2 forward."""
    import torch
    threads, tried, ncpu = pick_cpu_threads(probe)
    torch.set_num_threads(threads)
    cfg, params, inp = _oracle_setup()
    for _ in range(max(1, warmup)):
        cpu_oracle_step(params, inp, cfg)                    # warm-up
    ts = []
    for _ in range(iters):
        t0 = time.perf_counter()
        cpu_oracle_step(params, inp, cfg)
        ts.append(time.perf_counter() - t0)
    return ts, threads


def time_cpu_oracle_train():
    """The reference CPU training step stand-in: oracle forward (train mode) + torch.autograd backward at C2 on the
    host cores (clip + Adam omitted: <1 % of the step).  One warm-up + one timed step (~5-15 s each)."""
    import torch
    from oracle import tacotron_oracle as O
    threads = pick_cpu_threads(False)[0]
    torch.set_num_threads(threads)
    cfg = O.OracleConfig(r=R)
    params = O.init_params(cfg, seed=1)
    inp = O.synthetic_inputs(cfg, B, TX, T, seed=0)
    enc_m, dec_m = O.dropout_masks(cfg, B, TX, T, seed=2)
    sm = O.sched_mask(cfg, B, T, seed=3)
    ts = []
    for _ in range(2):
        t0 = time.perf_counter()
        O.loss_and_grads(params, inp, cfg, enc_drop_masks=enc_m, dec_drop_masks=dec_m, sample_mask=sm)
        ts.append(time.perf_counter() - t0)
    return ts[-1], threads


def measure_cpu_reference(steps, warmup, probe):
    """The CPU arm on ALL the host cores it can use.  (1) one process, threads probed ({16,32,64}) or 16; (2) the C2 batch
    sharded over processes x that many threads (logical CPUs, then physical cores), each layout tried for 2 steps; the
    fastest layout is then timed for `steps` steps.  Returns value (frames/s), sec_per_step and the cpu_baseline object."""
    ts, threads = time_cpu_oracle(steps, warmup=warmup, probe=probe)
    _, tried, ncpu = pick_cpu_threads(probe)
    sec = statistics.mean(ts)
    single = {"processes": 1, "threads": threads, "sec_per_step": sec}
    layout = dict(single)
    sharded = []
    th_s = threads if ncpu >= 2 * threads else max(1, ncpu // 2)
    cands = []
    for nsh in (ncpu // th_s, ncpu // (2 * th_s)):           # all logical CPUs, then one thread per physical core (2-way SMT)
        nsh = min(nsh, B)
        while nsh > 1 and B % nsh:
            nsh -= 1
        if nsh > 1 and nsh not in cands:
            cands.append(nsh)
    best_probe = None
    for nsh in cands:
        sps = time_cpu_oracle_sharded(2, 1, nsh, th_s)
        sharded.append({"processes": nsh, "threads": th_s, "sec_per_step_2_steps": sps})
        if sps is not None and (best_probe is None or sps < best_probe[1]):
            best_probe = (nsh, sps)
    if best_probe is not None and best_probe[1] < sec:
        sps = time_cpu_oracle_sharded(steps, warmup, best_probe[0], th_s)
        if sps is not None and sps < sec:
            layout = {"processes": best_probe[0], "threads": th_s, "sec_per_step": sps}
    sec = layout["sec_per_step"]
    cpu = {"value": FRAMES / sec, "unit": "mel frames/s", "cores": layout["processes"] * layout["threads"], "kind": "port",
           "host_cpus": ncpu, "layout": layout, "single_process": single, "sharded_probes": sharded,
           "threads_probed_sec_per_step": tried,
           "sample": f"{steps} full C2 forward passes (32000 frames each) after {warmup} warm-up, mean; the batch is sharded over "
                     f"processes when that is faster (utterances are independent in inference)"}
    return {"value": FRAMES / sec, "sec_per_step": sec, "cpu_baseline": cpu}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  TensorFlow 1.2 cannot be installed here
    (Python 3.12, no network; DESIGN.md section 5), so this is the oracle port (`kind: "port"`), all host threads it can
    use (probed), same metric / config keys / steps / warm-up as our arm; each step = one full C2 forward (about 1 s)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, args.steps)
    warmup = max(args.warmup, 1)
    m = measure_cpu_reference(steps, warmup, probe=True)
    val, sec = m["value"], m["sec_per_step"]
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "mel frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_dict(args.gpus),
        "run": {"precision": "fp32 (PyTorch CPU, MKL/oneDNN)", "cuda_graph": False},
        "note": "reference arm = CPU oracle port of the TF-1.2 graph (TF 1.2 not installable: py3.12, no network)",
        "cpu_baseline": m["cpu_baseline"],
        "e2e": {"value": val, "unit": "mel frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


_T0 = time.perf_counter()


def _log(msg):
    """progress on stderr (stdout carries only the JSON line)"""
    sys.stderr.write(f"[bench {time.perf_counter() - _T0:7.1f}s] {msg}\n")
    sys.stderr.flush()


def measure_train(args, world, rank, n=5, warm=2):
    """Side measurement (SURVEY.md section 8d(ii), 8e): the TRAINING step on the same C2 batch per rank -- train-mode
    forward (dropout, scheduled sampling 0.5), L1 losses, hand-written backward, one SUM all-reduce of the flat
    28.4 MB gradient bucket over NCCL when N > 1 (config C4 = N x C2), global-norm clip, Adam.  Never allowed to break
    the headline line: every rank first proves its own step works WITHOUT the collective, the ranks agree on that
    (MIN all-reduce of a flag), and only then are the data-parallel steps run and timed."""
    import torch
    import torch.distributed as dist
    from tacotron_b200 import Config, Tacotron
    from tacotron_b200.utils import dist as D
    ok, err, m, gi = 1, None, None, None
    try:
        cfg = Config(r=R, vocab_size=64, precision=args.precision)
        m = Tacotron(cfg, None, train=True, seed=1)
        g = torch.Generator().manual_seed(100 + rank)
        gi = {"text": torch.randint(1, 64, (B, TX), generator=g, dtype=torch.int32).cuda(),
              "text_length": torch.full((B,), TX, dtype=torch.int32).cuda(),
              "mel": torch.randn(B, T, 80 * R, generator=g).half().float().cuda(),
              "stft": torch.randn(B, T, 1025 * R, generator=g).half().float().cuda()}
        m.dp = False
        m.train_step(gi, lr=1e-4)                          # local step: no collective
        torch.cuda.synchronize()
        if not math.isfinite(float(m.loss)):
            raise RuntimeError("non-finite training loss")
    except Exception as ex:
        ok, err = 0, f"{type(ex).__name__}: {str(ex)[:160]}"
    if world > 1:
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        all_ok = int(flag.item())
    else:
        all_ok = ok
    if not all_ok:
        return {"error": err or "another rank failed its local training step"}
    try:
        m.dp = True
        for _ in range(max(warm, 2)):
            m.train_step(gi, lr=1e-4)
        D.barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        ev[0].record()
        for i in range(n):
            m.train_step(gi, lr=1e-4)
            ev[i + 1].record()
        torch.cuda.synchronize()
        D.barrier()
        ms = D.max_over_ranks(ev[0].elapsed_time(ev[n]) / n)
        loss = float(m.loss)
        # exposed communication: the same steps without the collective (every rank keeps stepping on its own gradients;
        # the parameters diverge across ranks from here on, nothing after this point exchanges them)
        exposed = None
        if world > 1:
            m.dp = False
            m.train_step(gi, lr=1e-4)
            D.barrier()
            ev2 = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            nl = min(n, 10)
            ev2[0].record()
            for i in range(nl):
                m.train_step(gi, lr=1e-4)
            ev2[1].record()
            torch.cuda.synchronize()
            D.barrier()
            ms_local = D.max_over_ranks(ev2[0].elapsed_time(ev2[1]) / nl)
            exposed = {"ms_per_step_without_allreduce": ms_local, "exposed_comm_ms": ms - ms_local}
        # one more step with events between its phases (this rank only; the phases overlap host work differently than
        # in the free-running loop above, so they need not add up to ms_per_step exactly)
        sections = None
        try:
            from tacotron_b200 import kernels as K
            from tacotron_b200.models import ops
            e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            torch.cuda.synchronize()
            e[0].record()
            S = {}
            with ops.saving(S):
                m.seq2seq_output, m.output = m.inference(gi, True)
            m.loss = m.add_loss_op(m.seq2seq_output, m.output, gi["mel"], gi["stft"])
            S.update(text=gi["text"], text_length=gi["text_length"], mel=gi["mel"], stft=gi["stft"])
            S["post/out"] = m.output
            e[1].record()
            m.backward(S)
            e[2].record()
            m._opt.apply(K, m.store.flat, 1e-4, m.config.cap_grads, allreduce=False)   # local: no collective outside the timed loop
            m.store.version += 1
            e[3].record()
            torch.cuda.synchronize()
            sections = {"forward_loss": e[0].elapsed_time(e[1]), "backward": e[1].elapsed_time(e[2]),
                        "sumsq_clip_adam": e[2].elapsed_time(e[3])}
        except Exception as ex:
            sections = {"error": f"{type(ex).__name__}: {str(ex)[:120]}"}
        return {"value": D.aggregate_throughput(FRAMES, world, ms), "unit": "mel frames/s", "ms_per_step": ms, "steps": n, "warmup": max(warm, 2) + 1,
                "n_gpus": world, "scaling": "weak",
                "config": f"training step on C2 per rank (B=32, char 128, T=200, r=5; global batch {32 * world}): dropout 0.5, scheduled "
                          "sampling 0.5, L1 losses, backward, clip 5, Adam; targets (2 x 141 MB) + activations exceed L2",
                "allreduce": ({"op": "SUM", "bytes_per_step": int(m.store.flat.numel() * 4), "backend": "nccl", **(exposed or {})} if world > 1 else None),
                "precision": (f"{args.precision} forward; backward fp32-grade: " +
                              ("exact-product FFMA GEMMs" if args.precision == "fp32" else "3xTF32 tensor-core GEMMs")),
                "loss_last_step": loss,
                "sections_ms": sections}
    except Exception as ex:
        return {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}


def measure_c5(args):
    """Side measurement, rank 0 only, no collective: BASELINE config 5 -- one utterance (B=1, prompt padded to 140
    chars, 500 mel frames = 100 decoder steps at r=5), inference through the public API with host text in and host
    waveform out, INCLUDING spectrogram inversion (Griffin-Lim, 50 iterations; audio.py:67-97, called at test.py:64).
    p50 over 20 runs.  The spectral-convergence self check guards against timing a broken inversion."""
    import torch
    from tacotron_b200 import Config, Tacotron, audio
    try:
        Bc, TXc, Tc = 1, 140, 100
        m = Tacotron(Config(r=R, vocab_size=64, max_decode_iter=Tc, precision=args.precision, cuda_graph=not args.no_graph), None,
                     train=False, seed=1)
        g = torch.Generator().manual_seed(0)
        text_h = torch.randint(1, 64, (Bc, TXc), generator=g, dtype=torch.int32).pin_memory()
        len_h = torch.full((Bc,), 97, dtype=torch.int32).pin_memory()
        n = 4 * R * (Tc // 4)
        wav_h = torch.empty((Bc, audio.hop_length * (n - 1)), dtype=torch.float32).pin_memory()
        mean = torch.full((1025 * R,), -4.0, device="cuda")          # stands in for the data set's stft_mean / stft_std
        std = torch.full((1025 * R,), 1.5, device="cuda")
        t_model, t_gl, t_all = [], [], []
        gl_mode = "eager (251 launches per inversion)"
        invert = lambda o: audio.invert_spectrogram(o, R, n_iter=50, stft_mean=mean, stft_std=std)
        if not args.no_graph:
            try:                                                     # the same kernels replayed from one CUDA graph
                glg = audio.GriffinLimGraph(Bc, Tc, R, n_iter=50)
                invert = lambda o: glg(o, stft_mean=mean, stft_std=std)
                gl_mode = "cuda-graph (1 launch per inversion)"
            except Exception as ex:
                gl_mode += f"; graph capture failed: {type(ex).__name__}: {str(ex)[:80]}"

        def once(record):
            t0 = time.perf_counter()
            ci = {"text": text_h.cuda(non_blocking=True), "text_length": len_h.cuda(non_blocking=True)}
            _, out = m.inference(ci, train=False)
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            wav = invert(out)
            wav_h.copy_(wav, non_blocking=True)
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            if record:
                t_model.append((t1 - t0) * 1e3); t_gl.append((t2 - t1) * 1e3); t_all.append((t2 - t0) * 1e3)
            return out, wav
        for _ in range(3):
            out, wav = once(False)
        for _ in range(20):
            out, wav = once(True)
        # self check: 50 iterations must have reduced || |STFT(y)| - mag ||_F / ||mag||_F well below the random-phase start
        mag = torch.exp(audio.reshape_frames(out[0], R, forward=False) * 1.5 - 4.0).t()          # [1025, n]
        win = torch.hann_window(audio.win_length, periodic=True, device="cuda")

        def conv(w):
            S = torch.stft(w, audio.n_fft, audio.hop_length, audio.win_length, window=win, center=True, pad_mode="reflect",
                           return_complex=True).abs()
            return float((S - mag).norm() / mag.norm())
        c50 = conv(wav[0])
        c0 = conv(audio.invert_spectrogram(out, R, n_iter=0, stft_mean=mean, stft_std=std)[0])
        return {"config": "C5: B=1, char 140, 500 mel frames (T=100, r=5), inference + Griffin-Lim x50 (n_fft 2048, win 1200, hop 300), "
                          "host text in, host waveform out", "p50_ms": statistics.median(t_all), "model_p50_ms": statistics.median(t_model),
                "griffinlim_p50_ms": statistics.median(t_gl), "griffinlim_mode": gl_mode, "runs": 20,
                "spectral_convergence": {"after_50": c50, "after_0": c0},
                "inversion_ok": bool(math.isfinite(c50) and c50 < c0)}
    except Exception as ex:
        return {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}


def measure_train_variant(args):
    """Child-process body (`--impl train-variant-worker`): the training step with each of taco_gemm's two kernels (3xTF32
    mma.sync = the model's choice in 'tf32' mode; exact-product FFMA = 'fp32' mode).  First the gradient of one C2 step is
    computed with both on identical saved activations (relative L2 difference reported), then 5 steps are timed with each."""
    import torch
    from tacotron_b200 import Config, Tacotron, kernels as K
    from tacotron_b200.models import ops
    try:
        cfg = Config(r=R, vocab_size=64, precision=args.precision)
        m = Tacotron(cfg, None, train=True, seed=1)
        g = torch.Generator().manual_seed(100)
        gi = {"text": torch.randint(1, 64, (B, TX), generator=g, dtype=torch.int32).cuda(),
              "text_length": torch.full((B,), TX, dtype=torch.int32).cuda(),
              "mel": torch.randn(B, T, 80 * R, generator=g).half().float().cuda(),
              "stft": torch.randn(B, T, 1025 * R, generator=g).half().float().cuda()}
        S = {}
        with ops.saving(S):
            m.seq2seq_output, m.output = m.inference(gi, True)
        S.update(text=gi["text"], text_length=gi["text_length"], mel=gi["mel"], stft=gi["stft"])
        S["post/out"] = m.output
        m.gemm_impl = 0                                    # exact-product FFMA kernel
        m.backward(S)
        g0 = m._opt.g.clone()
        m.gemm_impl = 1                                    # 3xTF32 mma.sync kernel (the model's choice in 'tf32' mode)
        m.backward(S)
        torch.cuda.synchronize()
        g1 = m._opt.g
        rel = float((g1 - g0).norm() / g0.norm())

        def timed(n=5):
            for _ in range(2):
                m.train_step(gi, lr=1e-4)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                m.train_step(gi, lr=1e-4)
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n
        ms_mma = timed()
        m.gemm_impl = 0
        ms_ffma = timed()
        res = {"note": "same training step with each GEMM kernel of the backward, one process, no collective",
               "grad_rel_l2_mma_vs_ffma": rel, "consistent": bool(rel < 1e-4),
               "mma_3xtf32": {"ms_per_step": ms_mma, "value": FRAMES / (ms_mma / 1e3), "unit": "mel frames/s"},
               "ffma_exact": {"ms_per_step": ms_ffma, "value": FRAMES / (ms_ffma / 1e3), "unit": "mel frames/s"}}
        print(json.dumps(res), flush=True)                 # keep this result even if the experimental route below faults
        return res
    except Exception as ex:
        return {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}


def _isolated(args, impl, limit):
    """run a side measurement in a child process with a time limit and return its JSON result"""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT",
                                                            "LOCAL_WORLD_SIZE", "GROUP_RANK", "ROLE_RANK", "TORCHELASTIC_RUN_ID")}
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", impl, "--precision", args.precision]
    if args.no_graph:
        cmd.append("--no-graph")
    try:
        out = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=limit)
        for ln in reversed(out.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": f"no result from the {impl} child (rc={out.returncode}): {out.stderr.strip()[-160:]}"}
    except subprocess.TimeoutExpired as te:
        txt = te.stdout.decode() if isinstance(te.stdout, bytes) else (te.stdout or "")
        for ln in reversed(txt.strip().splitlines()):      # keep what the child had already reported
            if ln.startswith("{"):
                r = json.loads(ln)
                r["child_note"] = f"child timed out after {limit} s; this is its last complete report"
                return r
        return {"error": f"{impl} child timed out ({limit} s)"}
    except Exception as ex:
        return {"error": f"{type(ex).__name__}: {str(ex)[:160]}"}


def measure_c5_isolated(args):
    """Runs measure_c5 in a child process (`bench.py --impl c5-worker`) with a time limit: the Griffin-Lim kernels have
    not had a hardware run yet (round 1), so neither a device fault nor a hang in them may touch the process that prints
    the headline line."""
    return _isolated(args, "c5-worker", 240)


DUMP_OUTPUT_SAMPLE = 8 * 1024 * 1024            # elements of `output` kept by --dump-outputs (32 MB of float32)


def dump_outputs(out_dir, y, out, align):
    """Write what one inference step returns to its caller as float32 .npy files: seq2seq_output [B, T, 80 r] (10 MB)
    and alignments [B, T, Tx] (3 MB) whole; of output [B, T, 1025 r] (131 MB) the flat elements at a fixed sorted random
    index set (torch.randperm, CPU generator seeded 0), so that all files stay under 64 MB together."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = out.reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_OUTPUT_SAMPLE].sort().values
    arrays = {"seq2seq_output": y, "alignments": align, "output_sample": flat[idx.to(flat.device)]}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tacotron_b200 import Config, Tacotron, _lib
    from tacotron_b200.utils import dist as D

    world, rank, local = D.world()
    torch.cuda.set_device(local)
    D.init("nccl")
    lib = _lib.lib()
    _log("torch + library loaded")

    cfg = Config(r=R, vocab_size=64, max_decode_iter=T, precision=args.precision, cuda_graph=not args.no_graph)
    model = Tacotron(cfg, None, train=False, seed=1)
    g = torch.Generator().manual_seed(rank)
    text_h = torch.randint(1, 64, (B, TX), generator=g, dtype=torch.int32).pin_memory()
    len_h = torch.full((B,), TX, dtype=torch.int32).pin_memory()
    inp = {"text": text_h.cuda(), "text_length": len_h.cuda()}
    model.step_ns = torch.zeros(T, dtype=torch.int64, device="cuda")
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")   # > 126 MB L2
    out_h = torch.empty((B, T, 1025 * R), dtype=torch.float32).pin_memory()
    align_h = torch.empty((B, T, TX), dtype=torch.float32).pin_memory()

    def step():
        return model.inference(inp, train=False)

    barrier = D.barrier

    # clocks are sampled from the first warm-up step to the end of the timed region (the GPU is under the
    # same load throughout; the timed region alone is too short for nvidia-smi's ~100 ms sampling period)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    _log("warm-up done (graphs captured)")
    t_warm = time.perf_counter()
    while sampler is not None and time.perf_counter() - t_warm < 0.35:      # keep the load on until a few samples exist
        step()
    barrier()

    # ---------------- device-resident timing: K steps, per-step events, L2 flushed between steps ----------------
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    dec_ms, enc_ms, post_ms, step_lat = [], [], [], []
    launches0 = lib.taco_launch_count()
    barrier()
    for i in range(args.steps):
        flush.zero_()
        model._marks = []
        starts[i].record()
        last = step()
        ends[i].record()
        marks = model._marks
        model._marks = None
        torch.cuda.synchronize()
        tt = {n: e for n, e in marks}
        enc_ms.append(tt["start"].elapsed_time(tt["encoder"]))
        dec_ms.append(tt["encoder"].elapsed_time(tt["decoder"]))
        post_ms.append(tt["decoder"].elapsed_time(tt["postnet"]))
        ns = model.step_ns.cpu().numpy()
        step_lat.extend(((ns[1:] - ns[:-1]) / 1e3).tolist())
    barrier()
    launches = lib.taco_launch_count() - launches0 + args.steps * int(model.last_graph_kernels)
    clocks = sampler.stop() if sampler else None
    _log("timed steps done")
    if args.dump_outputs and rank == 0:                  # before the e2e loop below overwrites the result buffers
        dump_outputs(args.dump_outputs, last[0], last[1], model.alignments)
        _log(f"outputs of the last timed step written to {args.dump_outputs}")
    total_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
    total_ms = D.max_over_ranks(total_ms)                 # the job advances at the slowest rank
    ms_per_step = total_ms / args.steps
    value = D.aggregate_throughput(FRAMES, world, ms_per_step)

    # ---------------- end to end through the public API with host buffers ----------------
    # Every step: H2D of the step's inputs from pinned memory, Tacotron.inference, D2H of output + alignments
    # into pinned memory.  The D2H of step i runs on a copy stream and overlaps the encoder/decoder of step
    # i+1 (the result buffers are only rewritten by the decoder / post-net sections, which wait for the copy).
    e2e_steps = args.steps                           # same step count as the device-timed region (the last D2H is not overlapped)
    copy_stream = torch.cuda.Stream()
    ev_done = torch.cuda.Event()
    ev_align_copied, ev_out_copied = torch.cuda.Event(), torch.cuda.Event()
    model.section_wait = {}
    barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        ci = {"text": text_h.cuda(non_blocking=True), "text_length": len_h.cuda(non_blocking=True)}
        y, out = model.inference(ci, train=False)
        ev_done.record()
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ev_done)
            align_h.copy_(model.alignments, non_blocking=True)
            ev_align_copied.record(copy_stream)
            out_h.copy_(out, non_blocking=True)
            ev_out_copied.record(copy_stream)
        model.section_wait = {"decoder": ev_align_copied, "postnet": ev_out_copied}
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    model.section_wait = None
    _log("e2e done")
    e2e_s = D.max_over_ranks((t1 - t0) / e2e_steps)
    e2e_val = D.aggregate_throughput(FRAMES, world, e2e_s * 1e3)
    h2d = text_h.numel() * 4 + len_h.numel() * 4
    d2h = out_h.numel() * 4 + align_h.numel() * 4

    train = None
    if not args.no_train:
        train = measure_train(args, world, rank)
        _log(f"training side measurement done: {train.get('ms_per_step', train.get('error'))}")

    if rank == 0:
        pk = peaks()
        dms = statistics.mean(dec_ms)
        ach = DECODER_GFLOP / dms                      # GFLOP / ms = TFLOP/s
        traffic = None
        for tp in ("r02_decoder_traffic.json", "r01_decoder_traffic.json"):     # ncu --set full capture of the same kernel (per launch)
            tp = os.path.join(ROOT, "profiles", tp)
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get("dram_bytes")
                break
        # the same step in the other precision modes, measured in the same run (5 steps each, this rank only):
        #   tf32 = single-pass TF32 tensor-core products (10-bit mantissa: NARROWER than the reference's fp32 arithmetic,
        #          stated tolerance 5e-3) -- a side result, never the headline;
        #   fp32 = exact-product FFMA kernel (the on-GPU cross-check path)
        def side_mode(prec, note):
            try:
                cfgp = Config(r=R, vocab_size=64, max_decode_iter=T, precision=prec, cuda_graph=not args.no_graph)
                mp = Tacotron(cfgp, None, train=False, seed=1)
                for _ in range(3):
                    mp.inference(inp, train=False)
                torch.cuda.synchronize()
                sp = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
                ep = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
                for i in range(5):
                    flush.zero_()
                    sp[i].record(); mp.inference(inp, train=False); ep[i].record()
                torch.cuda.synchronize()
                msp = sum(a.elapsed_time(b) for a, b in zip(sp, ep)) / 5
                del mp
                return {"value": FRAMES / (msp / 1e3), "unit": "mel frames/s", "ms_per_step": msp, "steps": 5, "note": note}
            except Exception as ex:           # never let a side measurement break the headline line
                return {"error": str(ex)[:200]}
        exact, tf32_mode = None, None
        if not args.no_fp32_mode:
            if args.precision != "tf32":
                tf32_mode = side_mode("tf32", "precision='tf32': single-pass TF32 products in the feed-forward contractions (parity "
                                              "tolerance 5e-3 of max|ref|, measured ~1e-3): narrower than the reference's fp32 -- side result only")
            if args.precision != "fp32":
                exact = side_mode("fp32", "precision='fp32': exact-product FFMA kernel for every feed-forward contraction (parity tolerance 2e-4)")
        _log("fp32-mode side measurement done")
        c5 = None if (args.no_c5 or world > 1) else measure_c5_isolated(args)     # single-GPU latency: N=1 runs only
        _log("C5 (single utterance + Griffin-Lim) side measurement done")
        if train is not None and "error" not in train and world == 1:
            train["gemm_kernels"] = _isolated(args, "train-variant-worker", 240)
            _log("training step with each GEMM kernel (child process) done")
        cpu = None
        if not args.no_cpu_baseline:
            try:
                cpu = measure_cpu_reference(3, 1, probe=False)["cpu_baseline"]
            except Exception as ex:                          # never lose the line over the side measurement: plain single-process timing
                ts, threads = time_cpu_oracle(3, warmup=1, probe=False)
                cpu = {"value": FRAMES / statistics.median(ts), "unit": "mel frames/s", "cores": threads, "kind": "port",
                       "host_cpus": os.cpu_count(), "sample": "3 full C2 forward passes of the PyTorch-CPU oracle (32000 frames each), median",
                       "note": f"layout probing failed: {type(ex).__name__}"}
            if train is not None and "error" not in train:
                try:
                    sec_t, thr_t = time_cpu_oracle_train()
                    train["cpu_baseline"] = {"value": FRAMES / sec_t, "unit": "mel frames/s", "cores": thr_t, "kind": "port",
                                             "sample": "1 C2 training step (forward + autograd backward) of the PyTorch-CPU oracle after 1 warm-up"}
                except Exception as ex:
                    train["cpu_baseline"] = {"error": str(ex)[:160]}
        _log("cpu baseline done")
        line = {
            "metric": METRIC, "value": value, "unit": "mel frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32x3": "f32", "tf32": "tf32", "fp32": "f32"}[args.precision],
            "dtype_note": {"fp32x3": "fp32-grade everywhere: feed-forward contractions = error-compensated 3xTF32 on tcgen05 (x = hi + lo; lo.hi + hi.lo + "
                                     "hi.hi, fp32 accumulate in TMEM; ~1e-6 relative), decoder = 3xTF32 mma.sync, bi-GRU = fp32 FFMA; passes the SAME "
                                     "tolerances as the exact-product FFMA mode (2e-5 per op, 2e-4 end to end vs the fp32 oracle)",
                           "tf32": "feed-forward contractions: single-pass TF32 tensor-core products, fp32 accumulate (tolerance 5e-3); recurrent kernels fp32-grade",
                           "fp32": "exact fp32 products (FFMA) in every feed-forward contraction"}[args.precision],
            "data": "synthetic",
            "config": config_dict(world),
            "run": {"precision": args.precision, "cuda_graph": not args.no_graph},
            "decoder_step_p50_us": statistics.median(step_lat) if step_lat else None,
            "sections_ms": {"encoder": statistics.mean(enc_ms), "decoder": dms, "postnet": statistics.mean(post_ms)},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": "mel frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_s * 1e3},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "decoder_kernel (persistent, 200 steps)", "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"],
                         "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"], "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read+write.sum)", "peak_source": pk["source"],
                         "algorithmic_gflop_per_launch": DECODER_GFLOP,
                         "whole_step": {"achieved": FWD_GFLOP / ms_per_step, "frac": FWD_GFLOP / ms_per_step / pk["bf16_tflops"]}},
            "tf32_mode": tf32_mode,
            "exact_fp32_mode": exact,
            "train": train,
            "c5_latency": c5,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception as ex:                            # teardown must never turn a printed result into a failed run
            _log(f"destroy_process_group: {ex}")


def run_train(args):
    """--mode train: the line's value is the C4 training step (N ranks x C2 per rank, global batch 32 N): train-mode
    forward, L1 losses, hand-written backward, ONE NCCL all-reduce (SUM) of the flat 28.4 MB gradient bucket, global-norm
    clip, Adam -- SURVEY.md section 8e.  Per-rank seeds; device-timed, max over ranks."""
    import torch
    import torch.distributed as dist
    from tacotron_b200 import _lib
    from tacotron_b200.utils import dist as D
    world, rank, local = D.world()
    torch.cuda.set_device(local)
    D.init("nccl")
    lib = _lib.lib()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = lib.taco_launch_count()
    tr = measure_train(args, world, rank, n=max(args.steps, 1), warm=max(args.warmup, 3))
    launches = lib.taco_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        ok = "error" not in tr
        line = {"metric": METRIC, "mode": "train", "value": tr.get("value"), "unit": "mel frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": tr.get("ms_per_step"), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if args.precision != "tf32" else "tf32", "data": "synthetic",
                "config": config_dict(world, workload=f"C4 synthetic: {world} x (B=32, char 128, 200 decoder steps, r=5) data-parallel TRAINING step "
                                                       "(dropout 0.5, scheduled sampling 0.5, L1 losses, backward, all-reduce, clip 5, Adam)",
                                      parallelism=f"dp{world}: one NCCL all-reduce (SUM) of the 28.4 MB gradient bucket per step",
                                      l2="targets (2 x 141 MB) + saved activations exceed L2 every step"),
                "run": {"precision": args.precision, "cuda_graph": False},
                "clocks": clocks, "gpu_launches": int(launches), "train": tr,
                "e2e": None}
        if not ok:
            line["error"] = tr["error"]
        print(json.dumps(line), flush=True)
    if world > 1:
        try:
            dist.destroy_process_group()
        except Exception:
            pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--threads", type=int, default=16, help="(internal: --impl reference-probe / reference-shard)")
    ap.add_argument("--nshards", type=int, default=1, help="(internal: --impl reference-shard)")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"],
                    help="infer (default, the BASELINE metric's configuration) or train: time the C4 data-parallel training step "
                         "(N x C2, one NCCL all-reduce of the 28.4 MB gradient bucket per step) as the line's value")
    ap.add_argument("--precision", default="fp32x3", choices=["fp32x3", "tf32", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fp32-mode", action="store_true", help="skip the side measurement of the exact-fp32 precision mode")
    ap.add_argument("--no-graph", action="store_true", help="launch kernels eagerly instead of replaying CUDA graphs")
    ap.add_argument("--no-train", action="store_true", help="skip the side measurement of the training step")
    ap.add_argument("--no-c5", action="store_true", help="skip the single-utterance + Griffin-Lim latency side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed inference step returned (rank 0) as DIR/<name>.npy, float32, < 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "infer"):
        ap.error("--dump-outputs applies to the default inference arm (--impl ours --mode infer) only")
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-probe":                 # internal: child process of pick_cpu_threads
        probe_worker(args.threads)
    elif args.impl == "reference-shard":                 # internal: child process of time_cpu_oracle_sharded
        shard_worker(args.threads, args.nshards, args.steps, args.warmup)
    elif args.mode == "train":
        run_train(args)
    elif args.impl == "c5-worker":                       # internal: child process of measure_c5_isolated
        print(json.dumps(measure_c5(args)), flush=True)
    elif args.impl == "train-variant-worker":            # internal: child process, opt-in GEMM kernel
        print(json.dumps(measure_train_variant(args)), flush=True)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
