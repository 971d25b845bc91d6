"""bench.py -- train-step throughput of the B200-native MIDIModel (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference|reference-gpu]
                    [--api fused|dropin] [--model tv2o-medium|tv2o-large|...] [--events S] [--batch B]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one full optimizer step in bf16 on a synthetic grammar-valid batch of (B per GPU, S+1 events,
8 tokens): embed -> event-level stack -> token-level stack -> lm_head -> CE (train.py:168-185) -> backward of all
of it -> [gradient all-reduce over NCCL when N > 1] -> global-norm clip + AdamW (train.py:121-138, 464).
Default workload = BASELINE.json configs[1]: tv2o-medium, B=8, S=2048.  Metric: MIDI-event tokens/s
(= global_batch * S * 8 / step time; all 8 token slots counted, pads included).

  value : device-timed (CUDA events, max over ranks), batches already resident in HBM
  e2e   : same step through the public API with the batch in pinned HOST memory: H2D copy of the
          batch and D2H read of the loss inside the timed region, every step
  roofline     : aggregate of all tcgen05 GEMM launches of the timed steps (CUDA events around each
                 launch on the launching stream): algorithmic FLOPs / measured time vs measured bf16 peak
  hbm_kernels  : the memory-bound kernels of the step (norm / RoPE / SwiGLU / CE / AdamW / sampler) timed alone on
                 bench-shape tensors: algorithmic bytes / time vs the measured copy bandwidth
  generate     : BASELINE's second metric, events/s of the KV-cached generate loop, with its HBM roofline
  cpu_baseline : the oracle port of the reference's path (fp32 eager PyTorch, host cores) on a
                 bounded sample (B=1, S=128 train step), rank 0 at N=1 only

--dump-outputs DIR (native arm, rank 0) writes what the last timed step computed as DIR/<name>.npy (float32): `loss`, and
`param.<name>` / `grad.<name>` for every trainable parameter after the optimizer update.  Inputs and weights are seeded, so
two builds run with the same arguments can be compared output for output -- to a tolerance: the order of the atomic
gradient accumulations varies, and two runs of one build already differ in the last bits.

Arms:
  --impl native (default)   this repo's kernels.  --api fused = MIDIModel.training_loss + fused_optimizer_step (the
                            headline); --api dropin = what UNCHANGED train.py gets: forward -> forward_token ->
                            F.cross_entropy -> loss.backward() -> clip_grad_norm_ -> torch AdamW (torch DDP at N > 1).
  --impl reference          the reference's CPU path (oracle port; the reference is pure Python and cannot travel).
  --impl reference-gpu      the reference's own GPU path on the same box: HF LlamaModel eager bf16 + torch SDPA +
                            F.cross_entropy + torch fused AdamW (midi_model.py:102-150, train.py:121-138,168-188) --
                            cuBLAS / ATen kernels only, nothing of this repo's engine.  The comparator the sm_100a
                            kernels have to beat (BASELINE.md section 4).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "midi-model_b200"), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ.pop("NCCL_DEBUG")           # (NCCL prints its version banner to stdout at VERSION and above: keep stdout
                                           #  to the single JSON line; an explicitly requested WARN / INFO is left alone)

import torch  # noqa: E402

METRIC = "train_tokens_per_sec"
UNIT = "MIDI-event tokens/s"
T_TOK = 8
LR, WARMUP_STEPS = 2e-4, 1000.0
DEFAULTS = {"model": "tv2o-medium", "events": 2048, "batch": 8, "task": "train"}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def model_dims(name: str):
    """(event-level layers, token-level layers): midi_model.py:71-75,92-94."""
    n = 24 if name.endswith("large") else 12
    return n, n // 4


def train_flops_per_token(model: str, S: int) -> float:
    """SURVEY.md Appendix C: forward 861.6 MFLOP/event for tv2o-medium at S=2048 (GEMMs + causal attention), x3."""
    H, V = 1024, 3406
    n_o, n_i = model_dims(model)
    outer = n_o * (4 * 2 * H * H + 3 * 2 * H * 4096 + 2 * 2 * H * (S + 1) / 2)
    inner = n_i * (4 * 2 * H * H + 3 * 2 * H * 1024 + 2 * 2 * H * (T_TOK + 1) / 2)
    per_event = outer + T_TOK * (inner + 2 * H * V)
    return 3.0 * per_event / T_TOK


def workload_name(args, what="train step (fwd+bwd+allreduce+clip+AdamW)"):
    return f"{args.model} {what} bf16, batch={args.batch}/GPU x {args.events} events x {T_TOK} tokens"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 - 0.1 <= t <= t1 + 0.3 and len(r) >= 7] or [r for _, r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        reasons = []
        for i, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
            if any(r[i].lower().startswith("active") for r in rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def dist_env():
    return int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))


def make_timed(world, dev, launch_counter=None):
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = launch_counter() if launch_counter else 0
        t0 = time.time()
        e0.record()
        for i in range(k):
            fn(i)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, (launch_counter() - l0 if launch_counter else 0), t0, time.time()

    return timed


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle's train step (fp32 eager PyTorch + torch AdamW), bounded sample
# ---------------------------------------------------------------------------------------------
def cpu_threads() -> int:
    # eager PyTorch at B=1 does not scale past a few dozen threads (profiles/r2_cpu_thread_sweep.txt: the 128-thread GPU
    # host is several times SLOWER with all threads than with 16): use up to 16 and report that count
    return min(os.cpu_count() or 1, int(os.environ.get("B200_CPU_THREADS", "16")))


def cpu_train_step_tokens_per_s(model_name: str, steps: int, warmup: int, batch: int = 1, n_events: int = 128):
    import midi_model as mm
    from midi_b200.synth import synth_batch
    from oracle import midi_oracle as O
    cores = cpu_threads()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.from_name(model_name)
    model = mm.MIDIModel(cfg)          # parameter container only; the arithmetic below is the oracle's
    ocfg = O.cfg_from_hf(cfg)
    params = dict(model.named_parameters())
    no_decay = [p for n, p in params.items() if "bias" in n or "norm" in n]
    decay = [p for n, p in params.items() if not ("bias" in n or "norm" in n)]
    opt = torch.optim.AdamW([dict(params=decay, weight_decay=0.01), dict(params=no_decay, weight_decay=0.0)], lr=LR,
                            betas=(0.9, 0.99), eps=1e-8)
    data = [synth_batch(model.tokenizer, batch, n_events + 1, seed=1234 + i) for i in range(2)]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        loss = O.train_loss(params, ocfg, data[i % 2])
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(list(params.values()), 1.0)
        opt.step()
        float(loss.detach())
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    tok = batch * n_events * T_TOK
    ms = 1e3 * sum(times) / len(times)
    return tok / (ms / 1e3), ms, cores, f"oracle fp32 train step (fwd+bwd+clip+AdamW), B={batch}, S={n_events}, {steps} steps after {warmup} warm-up"


def cpu_generate_events_per_s(model_name: str, n_events: int = 24):
    """The oracle's generate loop (midi_model.py:167-250 restated) on the host cores: b=1, default sampling, fp32."""
    import midi_model as mm
    from oracle import midi_oracle as O
    cores = cpu_threads()
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.from_name(model_name)
    model = mm.MIDIModel(cfg)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ocfg = O.cfg_from_hf(cfg)
    g = torch.Generator().manual_seed(1)
    done = 0
    t0 = time.perf_counter()
    with torch.no_grad():
        for attempt in range(8):       # seeded-init weights may emit EOS early: keep going until enough events were timed
            out = O.generate(sd, ocfg, model.tokenizer, None, batch_size=1, max_len=n_events + 1, generator=g)
            done += out.shape[1] - 1
            if done >= n_events:
                break
    dt = time.perf_counter() - t0
    return done / dt, cores, f"oracle fp32 generate(), batch 1, {done} events, temp=1.0 top_p=0.98 top_k=20"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    steps, warmup = args.steps, max(1, min(args.warmup, 2))
    v, ms, cores, sample = cpu_train_step_tokens_per_s(args.model, steps, warmup)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.model} train step, bounded CPU sample of batch={args.batch} x {args.events} events", "sample": sample},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------
# reference GPU arm: HF LlamaModel eager bf16 (the reference's own kernels: cuBLAS, ATen, SDPA)
# ---------------------------------------------------------------------------------------------
def run_reference_gpu(args):
    import torch.distributed as dist
    import torch.nn as nn
    import torch.nn.functional as F
    from transformers import LlamaModel
    import midi_model as mm                         # for MIDIModelConfig (presets + tokenizer tables) only
    from midi_b200.synth import synth_batch

    world, rank, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl reference-gpu needs a CUDA device")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = mm.MIDIModelConfig.from_name(args.model)
    tok = cfg.tokenizer

    class RefMIDIModel(nn.Module):
        """midi_model.py:102-150 as the reference wrote it: two HF LlamaModels + a Linear head."""

        def __init__(self):
            super().__init__()
            self.net = LlamaModel(cfg.net_config)
            self.net_token = LlamaModel(cfg.net_token_config)
            self.lm_head = nn.Linear(cfg.n_embd, tok.vocab_size, bias=False)

        def forward_token(self, hidden_state, x):
            hidden_state = hidden_state.unsqueeze(1)
            x = self.net_token.embed_tokens(x)
            x = torch.cat([hidden_state, x], dim=1)
            return self.lm_head(self.net_token(inputs_embeds=x, use_cache=False).last_hidden_state)

        def forward_events(self, x):
            x = self.net.embed_tokens(x).sum(dim=-2)
            return self.net(inputs_embeds=x, use_cache=False).last_hidden_state

        def forward(self, batch):                    # train.py:168-185
            x, y = batch[:, :-1].contiguous(), batch[:, 1:].contiguous()
            hidden = self.forward_events(x)
            hidden = hidden.reshape(-1, hidden.shape[-1])
            y = y.reshape(-1, y.shape[-1])
            logits = self.forward_token(hidden, y[:, :-1])
            return F.cross_entropy(logits.view(-1, tok.vocab_size), y.view(-1), reduction="mean", ignore_index=tok.pad_id)

    torch.manual_seed(0)
    model = RefMIDIModel().to(dev, dtype=torch.bfloat16).train()
    run = model
    if world > 1:
        from torch.nn.parallel import DistributedDataParallel as DDP
        run = DDP(model, device_ids=[local])
    named = list(model.named_parameters())
    no_decay = [p for n, p in named if "bias" in n or "norm" in n]
    decay = [p for n, p in named if not ("bias" in n or "norm" in n)]
    opt = torch.optim.AdamW([dict(params=decay, weight_decay=0.01), dict(params=no_decay, weight_decay=0.0)], lr=LR,
                            betas=(0.9, 0.99), eps=1e-8, fused=True)
    n_batches = 4
    host = [synth_batch(tok, args.batch, args.events + 1, seed=1234 + rank + 101 * i).pin_memory() for i in range(n_batches)]
    resident = [b.to(dev) for b in host]

    def step(batch_dev):
        loss = run(batch_dev)
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
        opt.step()
        return loss

    timed = make_timed(world, dev)
    W, K = max(3, args.warmup), max(1, args.steps)
    for i in range(W):
        step(resident[i % n_batches])
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    ms_total, _, t0, t1 = timed(lambda i: step(resident[i % n_batches]), K)
    losses = []

    def e2e_step(i):
        losses.append(float(step(host[i % n_batches].to(dev, non_blocking=True))))

    ms_e2e, _, _, t1 = timed(e2e_step, K)
    clocks = sampler.stop(t0, t1)
    tokens = world * args.batch * args.events * T_TOK
    pk, pk_kind = peaks()
    peak_tf = float(pk.get("bf16_tflops_sustained", 1400.0))
    step_tf = train_flops_per_token(args.model, args.events) * (args.batch * args.events * T_TOK) / (ms_total / K / 1e3) / 1e12
    line = {"impl": "reference-gpu", "metric": METRIC, "value": tokens / (ms_total / K / 1e3), "unit": UNIT, "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(args), "global_batch": world * args.batch, "n_events": args.events,
                       "tokens_per_event": T_TOK, "parallelism": f"dp{world}",
                       "kernels": "HF transformers LlamaModel eager bf16, torch SDPA, F.cross_entropy, torch fused AdamW, torch DDP"},
            "e2e": {"value": tokens / (ms_e2e / K / 1e3), "unit": UNIT, "ms_per_step": ms_e2e / K,
                    "h2d_bytes_per_step": int(host[0].numel() * host[0].element_size()), "d2h_bytes_per_step": 4,
                    "last_loss": losses[-1] if losses else None},
            "gpu_launches": 0, "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": step_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": step_tf / peak_tf,
                         "traffic": None, "kernel": "whole step (model FLOPs / step time)", "peak_kind": f"{pk_kind} sustained cuBLAS bf16"},
            "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


# ---------------------------------------------------------------------------------------------
# native arm
# ---------------------------------------------------------------------------------------------
def run_native(args):
    import torch.distributed as dist
    import torch.nn.functional as F
    import midi_model as mm
    from midi_b200 import lib, ops
    from midi_b200.synth import synth_batch

    world, rank, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib.load()
    B_PER_GPU, S_EVENTS = args.batch, args.events
    default_workload = all(getattr(args, k) == v for k, v in DEFAULTS.items())

    torch.manual_seed(0)                                   # identical seeded-init weights on every rank
    model = mm.MIDIModel(mm.MIDIModelConfig.from_name(args.model)).to(dev, dtype=torch.bfloat16).train()
    if args.task == "lora":
        # train.py --task lora (train.py:439-449): frozen base, rank-64 adapters on all seven projections of both stacks
        from midi_b200 import lora as _lora
        model.requires_grad_(False)
        model.add_adapter(_lora.LoraAdapterConfig(r=64, lora_alpha=128, lora_dropout=0, bias="none", task_type="CAUSAL_LM",
                                                  target_modules=["q_proj", "o_proj", "k_proj", "v_proj", "gate_proj",
                                                                  "up_proj", "down_proj"]))
    rt = model._rt()
    tok = model.tokenizer
    n_batches = 4
    host = [synth_batch(tok, B_PER_GPU, S_EVENTS + 1, seed=1234 + rank + 101 * i).pin_memory() for i in range(n_batches)]
    resident = [b.to(dev) for b in host]
    from midi_b200 import ddp
    state = {"step": 0}

    if args.api == "fused":
        # gradient averaging: NCCL all-reduce of the flat bf16 gradient buffer in 128 MB buckets on a side stream; the
        # token-level stack + lm_head slice is reduced while the event-level stack's backward is still running
        sync = ddp.GradSync(rt.store.gflat) if world > 1 else None

        def step(batch_dev):
            state["step"] += 1
            loss = model.training_loss(batch_dev, grad_ready=sync.ready if sync else None)
            if sync:
                sync.wait()
            lr = LR * min(1.0, state["step"] / WARMUP_STEPS)
            model.fused_optimizer_step(lr=lr, step=state["step"])
            return loss
    else:
        # what unchanged train.py runs (train.py:168-188, 121-138, 464; Lightning wraps the module in torch DDP)
        class Wrap(torch.nn.Module):
            def __init__(self, m):
                super().__init__()
                self.m = m

            def forward(self, batch):
                x, y = batch[:, :-1].contiguous(), batch[:, 1:].contiguous()
                hidden = self.m.forward(x)
                hidden = hidden.reshape(-1, hidden.shape[-1])
                y = y.reshape(-1, y.shape[-1])
                logits = self.m.forward_token(hidden, y[:, :-1])
                return F.cross_entropy(logits.view(-1, tok.vocab_size), y.view(-1), reduction="mean", ignore_index=tok.pad_id)

        run = Wrap(model)
        if world > 1:
            from torch.nn.parallel import DistributedDataParallel as DDP
            run = DDP(run, device_ids=[local])
        named = list(model.named_parameters())
        no_decay = [p for n, p in named if "bias" in n or "norm" in n]
        decay = [p for n, p in named if not ("bias" in n or "norm" in n)]
        opt = torch.optim.AdamW([dict(params=decay, weight_decay=0.01), dict(params=no_decay, weight_decay=0.0)], lr=LR,
                                betas=(0.9, 0.99), eps=1e-8, fused=True)

        def step(batch_dev):
            loss = run(batch_dev.to(torch.long))
            opt.zero_grad(set_to_none=True)
            loss.backward()
            torch.nn.utils.clip_grad_norm_(model.parameters(), 1.0)
            opt.step()
            return loss

    timed = make_timed(world, dev, lambda: lib.query("b200_launch_count"))
    W, K = max(3, args.warmup), args.steps
    for i in range(W):
        step(resident[i % n_batches])
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    last = {}

    def timed_step(i):
        last["loss"] = step(resident[i % n_batches])
    ms_total, launches, t0, t1 = timed(timed_step, K)      # the timed region (`value`)
    # taken before the passes below run more steps on the same model
    outputs = last_step_outputs(model, last["loss"]) if args.dump_outputs and rank == 0 else None
    # Roofline pass: the same K steps again with CUDA events around every GEMM launch.  It runs single-stream (the
    # weight-gradient GEMMs of the timed region run on a side stream under the HBM-bound kernels, where an event pair
    # would time the co-running kernels too), so `achieved` is each GEMM's own duration inside a full step.
    from midi_b200 import engine as _engine
    wg_stream, _engine.WGRAD_STREAM = _engine.WGRAD_STREAM, False
    ops.GEMM_PROFILE = []
    ms_prof, _, _, t1 = timed(lambda i: step(resident[i % n_batches]), K)
    prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
    _engine.WGRAD_STREAM = wg_stream
    clocks = sampler.stop(t0, t1)
    torch.cuda.synchronize()
    gemm_ms = sum(p[0].elapsed_time(p[1]) for p in prof)
    gemm_flops = sum(p[2] for p in prof)
    shapes = {}
    for e0, e1, fl, key in prof:
        ent = shapes.setdefault(key, [0, 0.0, 0.0])
        ent[0] += 1
        ent[1] += e0.elapsed_time(e1)
        ent[2] += fl
    per_shape = sorted(([*k, c, round(ms / K, 4), round(fl / (ms / 1e3) / 1e12, 1)] for k, (c, ms, fl) in shapes.items()),
                       key=lambda r: -r[-2])
    if rank == 0 and os.environ.get("B200_BENCH_VERBOSE"):
        print("M N K a_mn b_mn block_n splits count ms/step TF/s", file=sys.stderr)
        for r in per_shape:
            print(*r, file=sys.stderr)

    losses = []
    # end to end through the public API: int16 token batches in pinned host memory (the dataset's own dtype,
    # train.py:71) -> midi_b200.data.Prefetcher (H2D of batch i+1 on a copy stream while step i runs, inside the timed
    # region) -> MIDIModel.training_loss (widening + x/y split on the device) -> D2H read of the loss every step
    from midi_b200 import data as _data
    host16 = [_data.collate(list(h.numpy()), pad_id=0) for h in host]
    feed = iter(_data.Prefetcher((host16[i % n_batches] for i in range(K)), dev))

    def e2e_step(i):
        losses.append(float(step(next(feed))))              # D2H read of the loss

    ms_e2e, _, _, _ = timed(e2e_step, K)

    tokens_per_step = world * B_PER_GPU * S_EVENTS * T_TOK
    value = tokens_per_step / (ms_total / K / 1e3)
    e2e_value = tokens_per_step / (ms_e2e / K / 1e3)
    pk, pk_kind = peaks()
    peak_tf = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops", 1400.0)))
    ach_tf = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    step_tf = train_flops_per_token(args.model, S_EVENTS) * (B_PER_GPU * S_EVENTS * T_TOK) / (ms_total / K / 1e3) / 1e12
    if args.task == "lora":
        step_tf = 0.0          # the full-training FLOP model does not describe a LoRA step (no base weight gradients)

    api_note = ("MIDIModel.training_loss + fused_optimizer_step" if args.api == "fused" else
                "drop-in: forward -> forward_token -> F.cross_entropy -> backward -> clip_grad_norm_ -> torch fused AdamW (torch DDP at N>1)")
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": workload_name(args) if args.task == "train" else
                   workload_name(args, "LoRA train step (train.py --task lora: r=64, alpha=128, frozen base; fwd+bwd+allreduce+clip+AdamW over the adapters)"),
                   "api": api_note,
                   "global_batch": world * B_PER_GPU, "n_events": S_EVENTS, "tokens_per_event": T_TOK,
                   "parallelism": f"dp{world}", "weights": "seeded-init (torch.manual_seed(0))",
                   "l2": "per-step working set ~20 GB >> 126 MB L2 (no explicit flush needed); 4 distinct batches cycled"},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / K,
                "h2d_bytes_per_step": int(host16[0].numel() * host16[0].element_size()), "d2h_bytes_per_step": 4,
                "last_loss": losses[-1] if losses else None},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": ach_tf / peak_tf if peak_tf else None, "traffic": gemm_traffic() if default_workload else None,
                     "traffic_unit": "DRAM bytes (read+write) per GEMM launch, ncu capture of this command (profiles/*_gemm_traffic.json)",
                     "kernel": "gemm_tcgen05_kernel (every launch of K steps, CUDA events on the launching stream; single-stream pass of the same steps)", "peak_kind": f"{pk_kind} sustained cuBLAS bf16",
                     "gemm_ms_per_step": gemm_ms / K, "gemm_share_of_step": gemm_ms / ms_prof if ms_prof else None,
                     "profile_pass_ms_per_step": ms_prof / K, "wgrad_side_stream_in_timed_region": bool(wg_stream),
                     "whole_step_model_tflops": step_tf, "whole_step_frac": step_tf / peak_tf if peak_tf else None,
                     "per_shape": {"columns": "M,N,K,a_mn,b_mn,block_n,splits,launches,ms_per_step,TFLOP/s", "rows": per_shape}},
        "peak_mem_gb": torch.cuda.max_memory_allocated() / 2 ** 30,
    }
    if not args.no_hbm_kernels and default_workload:
        line["hbm_kernels"] = hbm_kernels_leg(model, dev, float(pk.get("hbm_gbs", 6586.4)), pk_kind)
    if not args.no_generate and default_workload:
        line["generate"] = generate_leg(model, dev, world, rank, float(pk.get("hbm_gbs", 6586.4)),
                                        cpu=(world == 1 and not args.no_cpu_baseline))
    if world == 1 and not args.no_cpu_baseline:
        v, ms, cores, sample = cpu_train_step_tokens_per_s(args.model, 3, 1)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "ms_per_step": ms}
    if outputs is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


DUMP_BUDGET_BYTES = 48 << 20


def last_step_outputs(model, loss):
    """The arrays a caller of the timed step holds after it: the loss, and every trainable parameter as the optimizer left
    it with the gradient that step computed.  A tensor larger than an equal share of DUMP_BUDGET_BYTES is reduced to a
    fixed, seeded sample of that many elements (the same positions for the parameter and its gradient)."""
    import numpy as np
    params = [(n, p) for n, p in model.named_parameters() if p.requires_grad]
    share = DUMP_BUDGET_BYTES // 4 // (2 * len(params))
    rng = np.random.default_rng(0)
    out = {"loss": loss.detach().float().cpu().numpy()}
    for name, p in params:
        idx = None
        if p.numel() > share:
            idx = torch.from_numpy(np.sort(rng.choice(p.numel(), share, replace=False))).to(p.device)
        for kind, t in (("param", p), ("grad", p.grad)):
            flat = t.detach().reshape(-1)
            out[f"{kind}.{name}"] = (flat if idx is None else flat[idx]).float().cpu().numpy()
    return out


def gemm_traffic():
    """DRAM bytes (read + write) per GEMM launch from the committed ncu capture of this same command (newest
    profiles/r*_gemm_traffic.json, derived from that round's launch list); None when no capture is committed."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_gemm_traffic.json")), reverse=True):
        try:
            with open(path) as f:
                return float(json.load(f)["dram_bytes_per_launch"])
        except (OSError, KeyError, ValueError):
            continue
    return None


def hbm_kernels_leg(model, dev, peak_gbs, pk_kind):
    """The memory-bound kernels of the path, each timed alone (CUDA events, 3 warm-up + 10 launches cycling through
    input sets larger than the 126 MB L2) on the tensors it sees in the benchmark step: achieved = algorithmic bytes
    (every operand read once + every result written once) / time, against the measured copy bandwidth."""
    from midi_b200 import decode as dec, lib, ops
    BF = torch.bfloat16
    H, V, pitch = 1024, 3406, 3408
    res = {"unit": "GB/s", "peak": peak_gbs, "peak_kind": f"{pk_kind} copy bandwidth", "kernels": {}}

    def run(name, make, fn, nbytes, sets):
        data = [make(i) for i in range(sets)]
        for i in range(3):
            fn(*data[i % sets])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for i in range(10):
            fn(*data[i % sets])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        gbs = nbytes / (ms * 1e-3) / 1e9
        res["kernels"][name] = {"us": round(ms * 1e3, 1), "bytes": int(nbytes), "gbs": round(gbs, 1), "frac": round(gbs / peak_gbs, 3)}
        del data

    g = torch.Generator(device=dev).manual_seed(0)
    rnd = lambda *s: torch.randn(*s, generator=g, device=dev, dtype=torch.float32).to(BF)
    w = (1 + 0.1 * rnd(H).float()).to(BF)
    for rows, tag, sets in ((16384, "event", 6), (131072, "token", 2)):
        run(f"add_rmsnorm_fwd[{tag} {rows}x1024]", lambda i: (rnd(rows, H), rnd(rows, H)),
            lambda x, r: ops.add_rmsnorm(x, r, w, 1e-6), rows * H * 2 * 4, sets)

        def mk_bwd(i):
            x = rnd(rows, H)
            return rnd(rows, H), x, torch.rsqrt(x.float().pow(2).mean(-1) + 1e-6), rnd(rows, H)
        dw = torch.empty(H, dtype=BF, device=dev)
        run(f"rmsnorm_bwd[{tag} {rows}x1024]", mk_bwd, lambda dy, x, rstd, dres: ops.rmsnorm_bwd(dy, x, w, rstd, dres, dw, False),
            rows * H * 2 * 4, sets)
    inter = {"event": 4096, "token": 1024}
    for rows, tag, sets in ((16384, "event", 2), (131072, "token", 1)):
        I = inter[tag]
        run(f"swiglu_fwd[{tag} {rows}x{I}]", lambda i: (rnd(rows, 2 * I),), lambda gu: ops.swiglu(gu), rows * I * 2 * 3, sets)
        run(f"swiglu_bwd[{tag} {rows}x{I}]", lambda i: (rnd(rows, 2 * I), rnd(rows, I)), lambda gu, da: ops.swiglu_bwd(gu, da),
            rows * I * 2 * 5, sets)
    inv = model.net.rotary_emb.inv_freq
    cos, sin = ops.rope_table(inv, 2048)
    run("rope_qk[event 16384x3072, q and k thirds in place]", lambda i: (rnd(16384, 3 * H),),
        lambda qkv: ops.rope_qk_(qkv, cos, sin, 2048, H, 64), 16384 * 2 * H * 2 * 2, 3)
    R = 131072
    tg = torch.randint(1, V, (R,), device=dev, generator=g)

    def mk_logits(i):
        t = torch.empty(R, pitch, dtype=BF, device=dev)
        t.normal_(generator=g)
        return (t,)
    holder = {}

    def ce_f(lg):
        holder["lac"], holder["lse"] = ops.ce_fwd(lg, tg, V, 0)
    run("ce_fwd[131072x3406]", mk_logits, ce_f, R * V * 2, 1)
    run("ce_bwd[131072x3406, in place]", mk_logits, lambda lg: ops.ce_bwd_(lg, tg, holder["lse"], holder["lac"], V, 0, 1.0),
        R * V * 2 * 2, 1)
    rt = model._rt()
    n = rt.store.numel
    st = model._opt_state(rt)
    parts = lib.query("b200_gradnorm_parts")
    ws = ops._ws("gradnorm", parts * 4, dev)

    def adamw():
        lib.call("b200_adamw_step", rt.store.flat.data_ptr(), rt.store.gflat.data_ptr(), st["m"].data_ptr(), st["v"].data_ptr(),
                 rt.store.nodecay.data_ptr(), n, 0.0, 0.9, 0.99, 1e-8, 0.0, 1, st["nc"].data_ptr(), lib.stream())
    run("adamw[233.8M params, lr=0]", lambda i: (), adamw, n * (2 + 2 + 4 + 4) + n * (2 + 4 + 4), 1)
    # fused sampler (temperature softmax + grammar range + top-p / top-k + draw) on one logits row per sequence
    glut = dec.GrammarLUT(model.tokenizer, dev)
    for Bs in (8, 1024):
        lg = torch.zeros(Bs, pitch, dtype=BF, device=dev)
        lg[:, :V] = rnd(Bs, V) * 2.5
        u = torch.rand(Bs, device=dev, generator=g)
        ev = torch.full((Bs,), model.tokenizer.event_ids["note"], dtype=torch.long, device=dev)
        outb = torch.zeros(Bs, 8, dtype=torch.long, device=dev)
        run(f"sample_from_logits[{Bs} rows x 3406, top_p .98 top_k 20]", lambda i: (),
            lambda: dec.sample_from_logits(lg, V, 1.0, 0.98, 20, 5, ev, glut, u, outb), Bs * V * 2, 1)
    return res


def generate_leg(model, dev, world, rank, peak_gbs, cpu=False):
    """BASELINE.json's second metric: events/s of the KV-cached generate loop (midi_model.py:167-250) with the
    reference's default sampling (temp 1.0, top-p 0.98, top-k 20), from one BOS event; replicas only across GPUs
    (each rank generates its own rows, no collective).  EOS stopping is disabled so the event count is fixed
    (seeded-init weights emit EOS at random).  Roofline (SURVEY.md 8d): HBM bytes one event step has to move =
    event-level layer weights + token-level layer weights + lm_head (the 8 token steps re-read theirs from L2) + the KV
    cache of the mean context, / measured copy bandwidth."""
    import torch.distributed as dist
    from midi_b200 import decode as dec
    rt = model._rt()
    tok = model.tokenizer
    res = {"unit": "events/s", "sampling": "temp=1.0 top_p=0.98 top_k=20", "note": "wall clock incl. launches, EOS stop disabled"}
    oc, ic = rt.outer.cfg, rt.inner.cfg
    w_outer = oc.n_layer * (4 * oc.hidden * oc.hidden + 3 * oc.hidden * oc.inner) * 2
    w_inner = ic.n_layer * (4 * ic.hidden * ic.hidden + 3 * ic.hidden * ic.inner) * 2 + rt.V * rt.H * 2
    # batch 8 runs BASELINE config 3 in full: 4096-event context (1 BOS + 4095 generated events per row)
    for B, n_new in ((1, 512), (8, 4095)):
        gg = dec.GraphGenerator(model._cached_stack("outer"), model._cached_stack("inner"), rt.lm_head, rt.pitch, rt.V, tok,
                                dec.GrammarLUT(tok, dev), B, n_new + 1, 1.0, 0.98, 20, 1234 + rank)
        prompt = torch.full((B, 1, tok.max_token_seq), tok.pad_id, dtype=torch.long, device=dev)
        prompt[:, 0, 0] = tok.bos_id
        def timed_run(mode):
            gg.run(prompt, use_graph=mode, check_every=1 << 30, stop_on_eos=False)      # warm-up (+ graph capture)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            out = gg.run(prompt, use_graph=mode, check_every=64, stop_on_eos=False)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if world > 1:
                t = torch.tensor([dt], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t.item())
            assert out.shape[1] == n_new + 1
            return dt
        dt_graph = timed_run(True)                 # one CUDA-graph replay (~210 kernel nodes) per event
        dt = timed_run("persist")                  # default: persistent cooperative kernel, 64 events per launch
        kv_bytes = oc.n_layer * B * (n_new / 2) * 2 * oc.hidden * 2            # K and V of the mean context, every layer
        step_bytes = w_outer + w_inner + kv_bytes
        ms = 1e3 * dt / n_new
        res[f"batch{B}"] = {"events_per_s": world * B * n_new / dt, "ms_per_event_step": ms, "rows": world * B,
                            "new_events_per_row": n_new, "loop": "persistent kernel (csrc/decode_persist.cu), 64 events per launch",
                            "graph_loop_events_per_s": world * B * n_new / dt_graph,
                            "roofline": {"bound": "hbm", "bytes_per_event_step": int(step_bytes),
                                         "achieved": step_bytes / (ms * 1e-3) / 1e9, "peak": peak_gbs, "unit": "GB/s",
                                         "frac": step_bytes / (ms * 1e-3) / 1e9 / peak_gbs,
                                         "events_per_s_at_roofline": B * peak_gbs * 1e9 / step_bytes}}
        del gg
    if cpu:
        v, cores, sample = cpu_generate_events_per_s("tv2o-medium")
        res["cpu_baseline"] = {"value": v, "unit": "events/s", "cores": cores, "kind": "port", "sample": sample}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "reference-gpu"])
    ap.add_argument("--api", default="fused", choices=["fused", "dropin"])
    ap.add_argument("--model", default=DEFAULTS["model"])
    ap.add_argument("--events", type=int, default=DEFAULTS["events"])
    ap.add_argument("--batch", type=int, default=DEFAULTS["batch"])
    ap.add_argument("--task", default=DEFAULTS["task"], choices=["train", "lora"], help="full training or LoRA (train.py:298)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-generate", action="store_true")
    ap.add_argument("--no-hbm-kernels", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs is implemented for --impl native")
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "reference-gpu":
        return run_reference_gpu(args)
    return run_native(args)


if __name__ == "__main__":
    sys.exit(main())
