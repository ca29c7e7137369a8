#!/usr/bin/env python
"""bench.py — coarse-stage training-step throughput of the B200-native hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo (torchrun launches it for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   # CPU arm: the oracle port of the reference path
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also write what the last timed step computed

With the same arguments every run sees the same inputs (seeded weights, token ids, dropout and mask draws), so the
files --dump-outputs writes can be compared between two builds of the project.

One "step" = one full optimiser step of the musiclm_small coarse stage (BASELINE.json configs[1]):
token pre-processing -> embedding gather -> 6 x (attention + conv-FFN) -> logit heads -> CE -> backward ->
gradient all-reduce (N > 1) -> global-norm clip -> AdamW, training semantics (FFN dropout 0.1 and the 15 %
forgetful mask active), batch 16 per GPU, N = 1024 positions, synthetic uniform token ids, random-init weights.
Prints ONE JSON line (rank 0).
"""
import argparse
import atexit
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TRAIN = dict(lr=3e-4, lr_warmup=6000, wd=0.01, max_grad_norm=0.5, ce_weights=[0.0, 0.0, 1.0])   # configs/training/*.json
COMMON = dict(dim=1024, attn_dropout=0.0, ff_dropout=0.1, grad_shrink_alpha=0.1)
# BASELINE.json configs[1..3] (SURVEY 8d): token shapes per sequence, per-GPU batch, N = positions fed to the transformer
WORKLOADS = {
    "cfg2": dict(stage="coarse", model=dict(depth=6, heads=8, num_coarse_quantizers=3), shapes=[(12,), (197,), (270, 3)], batch=16, N=1024, n_pred=811,
                 name="musiclm_small coarse-stage training step (BASELINE.json configs[1]): d=1024 L=6 h=8 conv-FFN F=2730, "
                      "N=1024 (clap 12 + semantic 197 + coarse 270x3)"),
    "cfg3": dict(stage="fine", model=dict(depth=6, heads=8, num_coarse_quantizers=3, num_fine_quantizers=5), shapes=[(12,), (254, 3), (1269,)], batch=8, N=2048,
                 n_pred=1270, name="musiclm_small fine-stage training step (BASELINE.json configs[2]): d=1024 L=6 h=8, N=2048 "
                                   "(clap 12 + coarse 254x3 + fine 1269 flattened: remainder heads), batch 8"),
    "cfg4": dict(stage="coarse", model=dict(depth=24, heads=16, num_coarse_quantizers=3), shapes=[(12,), (197,), (270, 3)], batch=16, N=1024, n_pred=811,
                 name="musiclm_large coarse-stage training step (BASELINE.json configs[3]: 16 per GPU, global 128 at 8 GPUs): "
                      "d=1024 L=24 h=16 conv-FFN F=2730, N=1024"),
}
METRIC = "coarse-stage training tokens/sec (positions fed to the transformer per optimiser step / step time)"
SEQ_N = WORKLOADS["cfg2"]["N"]


def synth_batch(B, gen, shapes=None):
    import torch
    shapes = shapes or WORKLOADS["cfg2"]["shapes"]
    return [torch.randint(0, 1024, (B,) + tuple(s), generator=gen) for s in shapes]


def make_model(wl):
    import open_musiclm_b200 as O
    fn = {"coarse": O.create_coarse_transformer, "fine": O.create_fine_transformer, "semantic": O.create_semantic_transformer}[wl["stage"]]
    return fn(**COMMON, **wl["model"])


def flops_per_step(B, N=SEQ_N, L=6, h=8, d=1024, n_pred=811):
    """ALGORITHMIC flops (SURVEY 8d): F = 2730 and C = 1025, not the padded tile sizes."""
    F = int(d * 8 / 3)
    G = 2 * d * (h * 64) + 2 * d * 128 + 2 * (h * 64) * d + 2 * d * 2 * F + 2 * F * d
    A = 2 * 64 * h * (N + 1)
    fwd_attn_ffn = B * N * L * (G + A)
    conv = B * N * L * 2 * 3 * 2 * F
    logits = B * n_pred * 2 * 1025 * d
    fwd = fwd_attn_ffn + conv + logits
    return dict(fwd_attn_ffn=fwd_attn_ffn, fwd=fwd, step=3 * fwd, gemm_fwd=B * N * L * G + logits)


def wl_flops(wl, B):
    return flops_per_step(B, N=wl["N"], L=wl["model"]["depth"], h=wl["model"]["heads"], n_pred=wl["n_pred"])


def cpu_model_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], burst=p["bf16_tflops"], sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]), src="measured")
    return dict(hbm_gbs=6650.0, burst=1590.0, sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        atexit.register(self._end)           # the sampler must not outlive a run that fails before stop()

    def _end(self):
        if self.p is not None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
            self.p = None
            return True
        return False

    def stop(self):
        sampled = self._end()
        self.f.flush(); self.f.seek(0)
        text = self.f.read()
        self.f.close()
        os.unlink(self.f.name)
        if not sampled:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        sm, mx, reasons = [], 0, set()
        for line in text.splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx = max(mx, float(c[2]))
            except ValueError:
                continue
            for name, val in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], c[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        load = [x for x in sm if x > 0.5 * mx] or sm
        med = load[len(load) // 2] if load else None
        return dict(sm_mhz=med, sm_max_mhz=mx or None, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------ CPU arm
def usable_cores():
    """Cores this process may actually use: scheduler affinity capped by the cgroup CPU quota (a container on a
    128-core host often owns far fewer; asking torch for all visible cores then oversubscribes and crawls)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return max(1, n)


def pick_cpu_threads():
    """Thread count with the best measured fp32 matmul throughput on this host (a few seconds of calibration on an
    FFN-shaped product), so the CPU arm uses 'all the host threads it can use' rather than all it can see."""
    import torch
    top = usable_cores()
    cands = sorted({c for c in (top, top // 2, top // 4, 64, 32, 16, 8) if 1 <= c <= top}, reverse=True)
    a, b = torch.randn(2048, 1024), torch.randn(1024, 2730)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        a @ b
        t0 = time.perf_counter()
        for _ in range(3):
            a @ b
        t = time.perf_counter() - t0
        if t < best_t * 0.95:
            best, best_t = c, t
    return best


def cpu_reference_arm(steps, warmup, budget_s=150.0):
    """The reference's own CPU path, as restated by the oracle (kind "port": /root/reference cannot travel to the
    GPU box): full coarse training step (forward, backward, clip 0.5, AdamW) in fp32 on all host cores, on a
    bounded sample of the workload (batch 2 instead of 16; CPU throughput is batch-linear)."""
    import numpy as np
    import torch
    from oracle import restatement as R
    cores = pick_cpu_threads()
    torch.set_num_threads(cores)
    cfg = R.coarse_cfg(ce_weights=TRAIN["ce_weights"])
    params = {k: v for k, v in R.init_state(cfg, seed=0).items()}
    names = [k for k in params if not k.endswith("beta")]
    state = {}
    gen = torch.Generator().manual_seed(1234)
    Bs = 2

    def one_step(it):
        toks = [t.numpy() for t in synth_batch(Bs, gen)]
        sd = {k: (v.clone().requires_grad_(True) if k in names else v) for k, v in params.items()}
        rng = np.random.default_rng(it)
        fm = R.forgetful_mask((Bs, SEQ_N), cfg.mask_prob, rng.standard_normal((Bs, SEQ_N)).astype(np.float32))
        keeps = [torch.from_numpy(rng.random((Bs, SEQ_N, cfg.ff_inner)) >= cfg.ff_dropout) for _ in range(cfg.depth)]
        loss = R.loss_and_logits(cfg, sd, toks, forget_mask=fm, drop_keeps=keeps)[0]
        loss.backward()
        grads = {k: sd[k].grad for k in names}
        with torch.no_grad():
            p = {k: params[k] for k in names}
            R.clip_and_adamw(p, grads, state, step=it, lr=TRAIN["lr"], wd=TRAIN["wd"], max_grad_norm=TRAIN["max_grad_norm"],
                             warmup_iters=TRAIN["lr_warmup"])
        return float(loss)

    t_first = time.perf_counter(); one_step(0); t_first = time.perf_counter() - t_first
    warm_left = max(0, warmup - 1)
    # keep the whole run within the budget: cap the number of timed steps if a step is slow on this host
    est = max(t_first * 0.6, 1e-3)
    steps_eff = max(1, min(steps, int((budget_s - t_first) / est) - warm_left))
    for i in range(min(warm_left, 2)):
        one_step(1 + i)
    times = []
    for i in range(steps_eff):
        t0 = time.perf_counter(); one_step(10 + i); times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return dict(tokens_per_s=Bs * SEQ_N / med, ms_per_step=med * 1e3, cores=cores, steps=steps_eff,
                sample=f"oracle port of the reference training step (fwd+bwd+clip+AdamW, fp32, dropout+forgetful mask on), "
                       f"batch {Bs} x N {SEQ_N} (1/8 of the GPU batch), median of {steps_eff} steps after warm-up")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_arm(args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["tokens_per_s"], "unit": "tokens/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "musiclm_small coarse-stage training step, N=1024 (BASELINE.json configs[1]), CPU sample batch 2"},
        "cpu_baseline": {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "cpu_model": cpu_model_name(), "kind": "port", "sample": r["sample"]},
        "e2e": {"value": r["tokens_per_s"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
class Instrument:
    """Kernel-launch accounting and one CUDA-event pair per GEMM-family launch (off during the timed regions)."""
    kernels_per_call = {"omlm_attn_bwd": 2, "omlm_attn_bwd_tc": 2, "omlm_ffn_mid_bwd": 2}

    def __init__(self):
        import torch
        from open_musiclm_b200 import lib
        import open_musiclm_b200.engine as eng_mod
        self.torch, self.lib = torch, lib
        self.launches, self.on, self.log, self.dims = 0, False, [], {}
        orig_call, orig_gemm, orig_up = lib.call, lib.gemm, lib.gemm_ffn_up

        def counting_call(name, *a):
            self.launches += self.kernels_per_call.get(name, 1)
            return orig_call(name, *a)

        def alg(v):       # padded tile dimension -> the algorithmic one (Fp -> F, 2 Fp -> 2 F, Cp -> C)
            return self.dims.get(v, v)

        def timed_gemm(a, b, out, **kw):
            if not self.on:
                return orig_gemm(a, b, out, **kw)
            a_mn, b_mn = kw.get("a_mn", False), kw.get("b_mn", False)
            M = kw.get("M") or (a.shape[1] if a_mn else a.shape[0])
            K = kw.get("K") or (a.shape[0] if a_mn else a.shape[1])
            Nn = kw.get("N") or (b.shape[1] if b_mn else b.shape[0])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = orig_gemm(a, b, out, **kw); e1.record()
            self.log.append((e0, e1, 2.0 * alg(M) * alg(Nn) * alg(K)))
            return r

        def timed_ffn_up(xn, w1p, cwp, u, h, rowsum, Nseq, Fp, **kw):   # the FFN-up GEMM (conv + GEGLU fused in its epilogue)
            if not self.on:
                return orig_up(xn, w1p, cwp, u, h, rowsum, Nseq, Fp, **kw)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); r = orig_up(xn, w1p, cwp, u, h, rowsum, Nseq, Fp, **kw); e1.record()
            self.log.append((e0, e1, 2.0 * xn.shape[0] * alg(2 * Fp) * xn.shape[1]))
            return r
        lib.call = counting_call
        lib.gemm = eng_mod.lib.gemm = timed_gemm
        lib.gemm_ffn_up = eng_mod.lib.gemm_ffn_up = timed_ffn_up

    def set_dims(self, eng):
        self.dims = {eng.Fp: eng.F, 2 * eng.Fp: 2 * eng.F}
        for c, cp in zip(eng.C, eng.Cp):
            self.dims[cp] = c


def measure(key, args, world, rank, local, inst, full):
    """Times one workload.  full: the headline treatment (e2e loop, per-launch GEMM events, forward-only, re-check);
    otherwise device-timed steps + forward only (the other BASELINE configs reported beside the headline)."""
    import torch
    import torch.distributed as dist
    import open_musiclm_b200 as O
    wl = WORKLOADS[key]
    B = args.batch if (full and args.batch) else wl["batch"]
    steps = args.steps
    torch.manual_seed(0)                                      # identical init on every rank (= the reference's init)
    model = make_model(wl).cuda()
    tr = O.HotPathTrainer(model, cross_entropy_loss_weights=TRAIN["ce_weights"], lr=TRAIN["lr"], lr_warmup=TRAIN["lr_warmup"],
                          wd=TRAIN["wd"], max_grad_norm=TRAIN["max_grad_norm"], grad_accum_every=1, seed=rank)
    inst.set_dims(tr.eng)
    gen = torch.Generator().manual_seed(1234 + rank)
    pool_host = [[t.pin_memory() for t in synth_batch(B, gen, wl["shapes"])] for _ in range(8)]
    pool_dev = [[t.cuda() for t in b] for b in pool_host]
    h2d = sum(t.numel() * t.element_size() for t in pool_host[0])

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n, finish=None):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        if finish is not None:
            finish()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / n

    step_dev = lambda i: tr.train_step([pool_dev[i % len(pool_dev)]])
    # first step: eager launches, counted (the CUDA graph captured two steps later replays exactly these kernels)
    inst.launches = 0
    step_dev(0)
    n_launch = inst.launches
    for i in range(max(args.warmup, 3)):
        step_dev(i + 1)
    sampler = ClockSampler(local) if (full and rank == 0) else None
    if sampler:
        sampler.start()
    ms_step = timed(step_dev, steps)
    fl = wl_flops(wl, B)
    peaks = load_peaks()
    tok = world * B * wl["N"]
    res = dict(key=key, B=B, tok=tok, ms_step=ms_step, n_launch=n_launch, fl=fl, steps=steps, h2d=h2d, tr=tr)
    if full:
        # end to end through the public trainer API: every step copies its batch from pinned host memory and its loss back
        # to the host; the loss of step i is read on the host while step i+1 runs (one-step logging lag), the last one
        # before the timed region closes
        pending, host_losses = [], []

        def step_e2e(i):
            pending.append(tr.train_step_async([pool_host[i % len(pool_host)]]))
            if len(pending) > 1:
                host_losses.append(pending.pop(0).value())

        def drain_e2e():
            while pending:
                host_losses.append(pending.pop(0).value())
        for i in range(2):
            step_e2e(i)
        drain_e2e()
        host_losses.clear()
        res["ms_e2e"] = timed(step_e2e, steps, finish=drain_e2e)
        assert len(host_losses) == steps and all(math.isfinite(v) for v in host_losses), "e2e: every step's loss must reach the host"
        res["clocks"] = sampler.stop() if sampler else None
        # ---- instrumented steps: GEMM family (the dominant kernel) with one CUDA-event pair per launch
        graph_was = tr.use_cuda_graph
        tr.use_cuda_graph = False            # per-launch CUDA events need eager launches (same kernels, same order)
        step_dev(0)
        inst.log.clear()
        inst.on = True
        res["ms_instr"] = timed(step_dev, steps)
        inst.on = False
        tr.use_cuda_graph = graph_was
        torch.cuda.synchronize()
        res["g_ms"] = sum(e0.elapsed_time(e1) for e0, e1, _ in inst.log)
        res["g_fl"] = sum(f for _, _, f in inst.log)
        res["n_gemm"] = len(inst.log) // steps
    # forward-only (attention + FFN + heads, eval): the north_star's forward roofline figure
    fwd_fn = lambda i: tr.eval_loss(pool_dev[i % len(pool_dev)])
    for i in range(3):
        fwd_fn(i)
    res["ms_fwd"] = timed(fwd_fn, steps)
    if full:
        # order check: the device loop again, now after the e2e and instrumented loops (same K), to expose any
        # power-cap / clock drift between the first and the later timed regions
        for i in range(2):
            step_dev(i)
        res["ms_step_again"] = timed(step_dev, steps)
    res["graph"] = tr.use_cuda_graph
    res["overlap"] = getattr(tr, "allreduce_mode", None)
    res["peaks"] = peaks
    return res


def measure_generation(seconds=10, batch=1):
    """BASELINE.json configs[4]: semantic -> coarse -> fine generation of `seconds` of audio through the reference's
    sliding windows (open_musiclm.py:925-1031) on the KV-cache decode path, random-init musiclm_small stages, synthetic
    clap ids.  tokens/s = sampled tokens of the three streams / device time (CUDA events) of the SECOND run (the first
    one captures the per-quantizer CUDA graphs)."""
    import torch
    import open_musiclm_b200 as O
    torch.manual_seed(0)
    mk = dict(**COMMON, depth=6, heads=8)
    sem = O.create_semantic_transformer(**mk).cuda().eval()
    coa = O.create_coarse_transformer(**mk, num_coarse_quantizers=3).cuda().eval()
    fin = O.create_fine_transformer(**mk, num_coarse_quantizers=3, num_fine_quantizers=5).cuda().eval()
    mlm = O.MusicLM(semantic_transformer=sem, coarse_transformer=coa, fine_transformer=fin)
    g = torch.Generator().manual_seed(1234)
    clap = torch.randint(0, 1024, (batch, 12), generator=g).cuda()
    times = []
    for it in range(2):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        ac, s, c, f = mlm.generate_tokens(clap_token_ids=clap, output_seconds=seconds, return_all=True)
        e1.record()
        torch.cuda.synchronize()
        times.append((e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3))
    n_tok = batch * (s.shape[1] * s.shape[2] + c.shape[1] * c.shape[2] + f.shape[1] * f.shape[2])
    ms_dev, ms_wall = times[-1]
    return {"workload": f"configs[4]: musiclm_small semantic->coarse->fine generation of {seconds} s of audio, batch {batch}, KV-cache decode, "
                        "sliding windows of MusicLM.forward, random-init weights, synthetic clap ids",
            "tokens_in_output": n_tok, "streams": {"semantic": list(s.shape), "coarse": list(c.shape), "fine": list(f.shape)},
            "ms_device": ms_dev, "ms_wall": ms_wall, "ms_first_run_incl_graph_capture": times[0][1],
            "tokens_per_s": n_tok / (ms_wall * 1e-3), "audio_seconds_per_second": seconds / (ms_wall * 1e-3)}


def summary(res):
    """Sub-result for a BASELINE config reported beside the headline."""
    fl, pk = res["fl"], res["peaks"]
    tps = res["tok"] / (res["ms_step"] * 1e-3)
    return {"workload": WORKLOADS[res["key"]]["name"], "per_gpu_batch": res["B"], "seq_len": WORKLOADS[res["key"]]["N"],
            "tokens_per_s": tps, "ms_per_step": res["ms_step"], "steps": res["steps"],
            "step_tflops_per_gpu": fl["step"] / (res["ms_step"] * 1e-3) / 1e12,
            "step_frac_of_sustained_peak": fl["step"] / (res["ms_step"] * 1e-3) / 1e12 / pk["sustained"],
            "forward_ms": res["ms_fwd"], "forward_attn_ffn_frac_of_sustained_peak": fl["fwd_attn_ffn"] / (res["ms_fwd"] * 1e-3) / 1e12 / pk["sustained"],
            "forward_attn_ffn_frac_of_burst_peak": fl["fwd_attn_ffn"] / (res["ms_fwd"] * 1e-3) / 1e12 / pk["burst"],
            "gpu_launches_per_step": res["n_launch"]}


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun for N > 1"
    inst = Instrument()
    res = measure(args.config, args, world, rank, local, inst, full=True)
    tr = res.pop("tr")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, tr.loss_out, tr.transformer)
    extras = {}
    del tr
    torch.cuda.empty_cache()
    for key in [k for k in args.extra.split(",") if k and k != "none" and k != args.config]:
        r = measure(key, args, world, rank, local, inst, full=False)
        r.pop("tr")
        extras[key] = summary(r)
        torch.cuda.empty_cache()
    if "cfg5" in [k for k in args.extra.split(",")] or args.extra == "cfg3,cfg4":
        try:
            extras["cfg5"] = measure_generation()
        except Exception as e:            # the headline must still be printed
            extras["cfg5"] = {"error": f"{type(e).__name__}: {e}"}
        torch.cuda.empty_cache()
    gemm_traffic = {}
    try:   # DRAM bytes of the GEMM family from the committed ncu --set full capture (tools/ncu_summarize.py)
        gemm_traffic = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_gemm_traffic.json")))
    except (OSError, ValueError):
        try:
            gemm_traffic = json.load(open(os.path.join(ROOT, "profiles", "r01_ncu_gemm_traffic.json")))
        except (OSError, ValueError):
            pass
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        r = cpu_reference_arm(steps=3, warmup=1, budget_s=60.0)
        cpu = {"value": r["tokens_per_s"], "unit": "tokens/s", "cores": r["cores"], "cpu_model": cpu_model_name(), "kind": "port", "sample": r["sample"],
               "cfg1_forward": cpu_cfg1_forward(r["cores"])}
    if rank == 0:
        wl, fl, peaks = WORKLOADS[args.config], res["fl"], res["peaks"]
        ms_step, ms_fwd, tok, B = res["ms_step"], res["ms_fwd"], res["tok"], res["B"]
        ach = res["g_fl"] / (res["g_ms"] * 1e-3) / 1e12
        line = {
            "metric": METRIC, "value": tok / (ms_step * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "ms_per_step_recheck_after_e2e": res["ms_step_again"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16 (fp16 operands for the forward GEMMs on LayerNorm outputs x weights; fp32 accumulate)", "data": "synthetic",
            "config": {"workload": wl["name"] + ", dropout 0.1 + forgetful mask 0.15, AdamW + clip 0.5",
                       "global_batch": world * B, "per_gpu_batch": B, "seq_len": wl["N"], "parallelism": f"dp{world}",
                       "l2": "no explicit flush: one step touches > 3 GB of activations/weights, far above the 126 MB L2"},
            "e2e": {"value": tok / (res["ms_e2e"] * 1e-3), "unit": "tokens/s", "ms_per_step": res["ms_e2e"], "h2d_bytes_per_step": res["h2d"],
                    "d2h_bytes_per_step": 4,
                    "api": "HotPathTrainer.train_step_async: batch copied from pinned host memory every step, loss copied "
                           "to pinned host memory every step and read on the host one step later (last one inside the timed region)"},
            "gpu_launches": res["n_launch"] * args.steps, "gpu_launches_per_step": res["n_launch"],
            "launch_mode": ("step replayed from CUDA graphs; gradient all-reduce: " + str(res["overlap"])) if res["graph"] else "eager launches",
            "roofline": {"bound": "tensor", "kernel": "gemm_bf16_kernel + gemm_ffn_up_kernel (tcgen05; all operand-major variants; FFN-up time includes its fused conv+GEGLU epilogue)", "achieved": ach,
                         "peak": peaks["sustained"], "unit": "TFLOP/s", "frac": ach / peaks["sustained"], "frac_of_burst_peak": ach / peaks["burst"],
                         "flops": "algorithmic (F = 2730, C = 1025; padded tile columns not counted)",
                         "traffic": gemm_traffic.get("bytes_per_launch"), "traffic_unit": "bytes per launch (family average)", "traffic_source": gemm_traffic.get("source"),
                         "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['src']})",
                         "launches_per_step": res["n_gemm"], "gemm_ms_per_step": res["g_ms"] / args.steps,
                         "gemm_share_of_step": (res["g_ms"] / args.steps) / res["ms_instr"], "ms_per_step_instrumented": res["ms_instr"]},
            "step_model_flops": {"tflop_per_step_per_gpu": fl["step"] / 1e12, "achieved_tflops_per_gpu": fl["step"] / (ms_step * 1e-3) / 1e12,
                                 "frac_of_sustained_peak": fl["step"] / (ms_step * 1e-3) / 1e12 / peaks["sustained"]},
            "forward_only": {"ms": ms_fwd, "attn_ffn_tflops": fl["fwd_attn_ffn"] / (ms_fwd * 1e-3) / 1e12,
                             "attn_ffn_frac_of_peak": fl["fwd_attn_ffn"] / (ms_fwd * 1e-3) / 1e12 / peaks["sustained"],
                             "attn_ffn_frac_of_burst_peak": fl["fwd_attn_ffn"] / (ms_fwd * 1e-3) / 1e12 / peaks["burst"],
                             "attn_ffn_frac_of_nominal_2250": fl["fwd_attn_ffn"] / (ms_fwd * 1e-3) / 1e12 / 2250.0},
            "configs": extras,
            "clocks": res["clocks"],
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, loss, model, n_sample=1 << 22):
    """What the last timed training step hands its caller: the step's loss (loss.npy) and the updated parameters
    (parameters.npy: all of them, flattened and concatenated in named_parameters() order; beyond n_sample entries, the
    entries at a fixed seeded sample of positions, in increasing order).  float32, 16 MB at most."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    with torch.no_grad():
        flat = torch.cat([p.detach().reshape(-1) for _, p in model.named_parameters()])
        if flat.numel() > n_sample:
            idx = torch.randint(0, flat.numel(), (n_sample,), generator=torch.Generator().manual_seed(0)).sort().values
            flat = flat[idx.to(flat.device)]
        np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())
        np.save(os.path.join(out_dir, "parameters.npy"), flat.float().cpu().numpy())


def cpu_cfg1_forward(cores):
    """BASELINE configs[0]: musiclm_small semantic-stage forward on the host cores, batch 2, N = 256 (oracle port, fp32,
    eval), median of 5 after 2 warm-ups."""
    import torch
    from oracle import restatement as R
    torch.set_num_threads(cores)
    cfg = R.semantic_cfg(ce_weights=[0.0, 1.0])
    sd = R.init_state(cfg, seed=0)
    g = torch.Generator().manual_seed(1234)
    toks = [torch.randint(0, 1024, (2, 12), generator=g).numpy(), torch.randint(0, 1024, (2, 241), generator=g).numpy()]
    ids, mask, _ = R.prepare_ids(cfg, toks, True, None)
    ts = []
    with torch.no_grad():
        for i in range(7):
            t0 = time.perf_counter(); R.forward_logits(cfg, sd, ids, mask); ts.append(time.perf_counter() - t0)
    ts = sorted(ts[2:])
    return {"tokens_per_s": 2 * 256 / ts[len(ts) // 2], "ms": ts[len(ts) // 2] * 1e3, "workload": "configs[0]: semantic forward, B=2, N=256, fp32"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch of the headline workload (0 = the config's own: 16 / 8 / 16)")
    ap.add_argument("--config", default="cfg2", choices=sorted(WORKLOADS), help="headline workload (default: BASELINE configs[1])")
    ap.add_argument("--extra", default="cfg3,cfg4", help="other BASELINE configs timed beside it (sub-results under 'configs'); 'none' to skip")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss and a fixed sample of the updated parameters "
                         "to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
