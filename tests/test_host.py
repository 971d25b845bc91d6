"""CPU-side tests: the C-ABI library loads and exports every symbol of include/midi_b200.h, the
drop-in module keeps the reference's contract, and the product refuses to run without CUDA."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _built():
    from midi_b200 import lib
    if not os.path.exists(lib.LIB_PATH):
        import subprocess
        import sys
        subprocess.check_call([sys.executable, os.path.join(ROOT, "midi-model_b200", "build_ext.py")])
    return lib


def test_library_exports_every_declared_symbol():
    lib = _built()
    hdr = open(os.path.join(ROOT, "include", "midi_b200.h")).read()
    declared = set(re.findall(r"\b(b200_\w+)\s*\(", hdr))
    assert len(declared) >= 30
    dll = ctypes.CDLL(lib.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(dll, s)]
    assert not missing, missing
    # the ctypes table mirrors the header one to one
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    lib.load()
    assert lib.query("b200_abi_version") == 1


def test_dropin_contract_and_seeded_init(golden_tiny):
    import midi_model as mm
    assert mm.config_name_list == ["tv1-medium", "tv2-medium", "tv2o-medium", "tv2-large", "tv2o-large"]
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64)
    m = mm.MIDIModel(cfg)
    sd = m.state_dict()
    for k, v in sd.items():      # same RNG consumption as the reference constructor => bit-identical weights
        np.testing.assert_array_equal(v.numpy(), golden_tiny["sd/" + k], err_msg=k)
    assert [n for n, _ in m.named_buffers()] == ["net.rotary_emb.inv_freq", "net.rotary_emb.original_inv_freq",
                                                "net_token.rotary_emb.inv_freq", "net_token.rotary_emb.original_inv_freq"]
    m16 = m.to(torch.bfloat16)
    np.testing.assert_array_equal(m16.net.rotary_emb.inv_freq.float().numpy(), golden_tiny["bf16/inv_freq_net"])


def test_medium_config_matches_reference_fixture(golden_medium):
    import midi_model as mm
    cfg = mm.MIDIModelConfig.from_name("tv2o-medium")
    assert cfg.tokenizer.vocab_size == 3406 and cfg.n_embd == 1024
    assert (cfg.net_config.num_hidden_layers, cfg.net_config.num_attention_heads, cfg.net_config.intermediate_size) == (12, 16, 4096)
    assert (cfg.net_token_config.num_hidden_layers, cfg.net_token_config.num_attention_heads,
            cfg.net_token_config.intermediate_size) == (3, 4, 1024)
    large = mm.MIDIModelConfig.from_name("tv2o-large")
    assert large.net_config.num_hidden_layers == 24 and large.net_token_config.num_hidden_layers == 6
    assert large.net_config.hidden_size == 1024       # reference: 2x layers only (SURVEY.md 0.7)
    with pytest.raises(ValueError):
        mm.MIDIModelConfig.from_name("tv3-medium")
    d = cfg.to_dict()
    cfg2 = mm.MIDIModelConfig(**{k: d[k] for k in ("tokenizer", "net_config", "net_token_config")})
    assert cfg2.net_config.hidden_size == 1024 and cfg2.tokenizer.vocab_size == 3406


def test_medium_seeded_init_and_oracle_golden(golden_medium):
    """The drop-in class regenerates the reference's seed-0 tv2o-medium weights; the oracle on them reproduces
    the reference's fp32 hidden / logits / loss fixture."""
    import midi_model as mm
    from oracle import midi_oracle as O
    g = golden_medium
    torch.manual_seed(0)
    m = mm.MIDIModel(mm.MIDIModelConfig.from_name("tv2o-medium"))
    sd = m.state_dict()
    assert len(sd) == int(g["n_tensors"]) == 140 and sum(v.numel() for v in sd.values()) == int(g["n_params"]) == 233842688
    for k in [k[5:] for k in g if k.startswith("init/")]:
        v = sd[k].double()
        got = np.array([v.sum().item(), v.abs().sum().item(), v.flatten()[12345 % v.numel()].item()])
        np.testing.assert_allclose(got, g["init/" + k], rtol=1e-12)
    ocfg = O.cfg_from_hf(m.config)
    batch = torch.from_numpy(g["batch"])
    sd = {k: v.detach() for k, v in sd.items()}
    with torch.no_grad():
        h = O.forward(sd, ocfg, batch[:, :-1])
        lg = O.forward_token(sd, ocfg, h.reshape(-1, 1024), batch[:, 1:].reshape(-1, 8)[:, :-1])
        loss = O.train_loss(sd, ocfg, batch)
    np.testing.assert_allclose(h.reshape(-1, 1024).numpy()[:, :64], g["fp32/hidden"], rtol=2e-3, atol=2e-4)
    np.testing.assert_allclose(lg.numpy()[:, :, :128], g["fp32/logits"], rtol=2e-3, atol=2e-4)
    assert abs(h.double().norm().item() - float(g["fp32/hidden_norm"])) < 1e-3 * float(g["fp32/hidden_norm"])
    assert abs(loss.item() - float(g["fp32/loss"])) < 1e-4


def test_generate_signatures_follow_the_reference():
    """MIDIModel.generate = midi_model.py:167-168; MIDIModel.generate_stream = app.py:28-29 (the app's own loop)."""
    import inspect
    import midi_model as mm
    gen = list(inspect.signature(mm.MIDIModel.generate).parameters)[1:]
    assert gen == ["prompt", "batch_size", "max_len", "temp", "top_p", "top_k", "generator"]
    st = inspect.signature(mm.MIDIModel.generate_stream).parameters
    assert list(st)[1:] == ["prompt", "batch_size", "max_len", "temp", "top_p", "top_k", "disable_patch_change",
                            "disable_control_change", "disable_channels", "generator"]
    assert [st[k].default for k in list(st)[1:]] == [None, 1, 512, 1.0, 0.98, 20, False, False, None, None]
    assert inspect.isgeneratorfunction(inspect.unwrap(mm.MIDIModel.generate_stream)) or \
        inspect.isgeneratorfunction(mm.MIDIModel.generate_stream)


def test_collate_int16_matches_reference_collate_fn():
    """midi_b200.data.collate == train.py:82-86 (F.pad to the longest sample with pad_id, stack), kept in int16."""
    import torch.nn.functional as F
    from midi_b200 import data
    rng = np.random.default_rng(0)
    samples = [rng.integers(0, 3406, size=(n, 8)).astype(np.int16) for n in (5, 1, 9, 3)]
    got = data.collate(samples, pad_id=0, pin=False)
    ref = [torch.from_numpy(s.astype(np.int64)) for s in samples]                    # train.py:79-80
    mx = max(len(m) for m in ref)
    ref = torch.stack([F.pad(m, (0, 0, 0, mx - m.shape[0]), mode="constant", value=0) for m in ref])
    assert got.dtype == torch.int16 and got.shape == ref.shape
    assert torch.equal(got.to(torch.int64), ref)
    with pytest.raises(ValueError):
        data.collate([np.full((2, 8), 40000, dtype=np.int64)], pin=False)
    with pytest.raises(ValueError):
        data.collate([], pin=False)


def test_native_lora_merge(tmp_path):
    """load_merge_lora (midi_model.py:109-114) without peft: W += B @ A * alpha / r on every target Linear, nothing else
    touched; accepts train.py's save_peft key layout and peft's `base_model.model.` prefixed layout."""
    import json
    import midi_model as mm
    from safetensors.torch import save_file
    try:
        import peft  # noqa: F401
        pytest.skip("peft installed: the reference sequence is used instead of the native merge")
    except ImportError:
        pass
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64)
    m = mm.MIDIModel(cfg)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(1)
    r, alpha = 4, 8.0
    targets = ["net.layers.0.self_attn.q_proj", "net.layers.1.self_attn.v_proj", "net_token.layers.0.self_attn.q_proj"]
    w = {}
    for i, t in enumerate(targets):
        out_f, in_f = before[t + ".weight"].shape
        prefix = "base_model.model." if i == 1 else ""
        suffix = ".default" if i == 2 else ""
        w[f"{prefix}{t}.lora_A{suffix}.weight"] = torch.randn(r, in_f, generator=g) * 0.1
        w[f"{prefix}{t}.lora_B{suffix}.weight"] = torch.randn(out_f, r, generator=g) * 0.1
    save_file(w, str(tmp_path / "adapter_model.safetensors"), metadata={"format": "pt"})
    (tmp_path / "adapter_config.json").write_text(json.dumps(
        {"peft_type": "LORA", "r": r, "lora_alpha": alpha, "target_modules": ["q_proj", "v_proj"], "fan_in_fan_out": False}))
    merged = m.load_merge_lora(str(tmp_path))
    assert merged is m
    after = m.state_dict()
    keys = list(w)
    for i, t in enumerate(targets):
        A, B = w[keys[2 * i]], w[keys[2 * i + 1]]
        np.testing.assert_allclose(after[t + ".weight"].numpy(), (before[t + ".weight"] + (B @ A) * (alpha / r)).numpy(),
                                   rtol=1e-6, atol=1e-7)
    touched = {t + ".weight" for t in targets}
    for k, v in after.items():
        if k not in touched:
            assert torch.equal(v, before[k]), k


def test_lazy_logits_routes_cross_entropy(monkeypatch):
    """SURVEY.md 8 f2 plumbing on CPU: the tensor forward_token returns in training is a dense logits tensor whose
    `F.cross_entropy(logits.view(-1, V), y, reduction="mean", ignore_index=pad)` (train.py:180-185) is served by the
    fused CE entry points on the pitched buffer, the gradient comes back as a view of that buffer, and every other use
    falls through to the ordinary dense path.  (The CE kernels themselves are replaced by torch stand-ins here; the GPU
    suite checks the real ones against the oracle through the same route.)"""
    import midi_model as mm
    import torch.nn.functional as F
    N, L, V, pitch = 3, 4, 10, 16
    calls = []

    def ce_fwd(buf, targets, V_, ignore):
        lg = buf[:, :V_].float()
        lse = torch.logsumexp(lg, -1)
        valid = targets != ignore
        nll = lse - lg.gather(1, targets.clamp_min(0)[:, None])[:, 0]
        cnt = valid.sum().float()
        calls.append("fwd")
        return torch.stack([(nll * valid).sum() / cnt, cnt]), lse

    def ce_bwd_(buf, targets, lse, lac, V_, ignore, grad_scale=1.0, grad_scale_dev=None):
        if grad_scale_dev is not None:
            grad_scale = grad_scale * float(grad_scale_dev)
        p = torch.exp(buf[:, :V_].float() - lse[:, None])
        p[torch.arange(p.shape[0]), targets] -= 1.0
        p[targets == ignore] = 0.0
        buf.data[:, :V_] = (p * (grad_scale / lac[1])).to(buf.dtype)     # raw write, like the kernel (no version bump)
        calls.append("bwd")

    monkeypatch.setattr(mm._ops, "ce_fwd", ce_fwd)
    monkeypatch.setattr(mm._ops, "ce_bwd_", ce_bwd_)
    torch.manual_seed(0)
    w = torch.randn(N * L, pitch).to(torch.bfloat16).requires_grad_(True)
    y = torch.randint(0, V, (N * L,))
    y[::5] = 0

    def make():
        buf = w * 1.0                                   # stands in for the lm_head GEMM output [N*L, pitch]
        return buf.view(N, L, pitch)[:, :, :V]

    ref = F.cross_entropy(make().reshape(-1, V).float(), y, reduction="mean", ignore_index=0)
    ref.backward()
    g_ref, w.grad = w.grad.clone(), None
    out = make()
    lz = out.as_subclass(mm.LazyLogits)
    lz._b200_lazy = (mm._as_pitched(out, N * L, pitch), V)
    hits = mm.LAZY_CE_HITS
    loss = F.cross_entropy(lz.view(-1, V), y.view(-1), reduction="mean", ignore_index=0)
    assert mm.LAZY_CE_HITS == hits + 1 and calls == ["fwd"]
    assert abs(float(loss) - float(ref)) < 2e-2
    loss.backward()
    assert calls == ["fwd", "bwd"]
    assert float((w.grad[:, :V].float() - g_ref[:, :V].float()).abs().max()) < 2e-3
    assert float(w.grad[:, V:].float().abs().max()) == 0.0
    # anything else is the ordinary dense tensor: slicing, argmax, a differently-configured loss
    w.grad = None
    lz2 = make().as_subclass(mm.LazyLogits)
    lz2._b200_lazy = (mm._as_pitched(lz2, N * L, pitch), V)
    assert torch.equal(torch.argmax(lz2, -1), torch.argmax(make(), -1))
    l_sum = F.cross_entropy(lz2.view(-1, V).float(), y, reduction="sum", ignore_index=0)
    assert mm.LAZY_CE_HITS == hits + 1                   # not intercepted
    l_sum.backward()
    assert w.grad is not None


def test_pitched_view_detection():
    """_as_pitched only accepts a [..., V] view that enumerates the rows of a [rows, pitch] bf16 buffer from its base."""
    import midi_model as mm
    buf = torch.zeros(12, 16, dtype=torch.bfloat16)
    v3 = buf.view(3, 4, 16)[:, :, :10]
    got = mm._as_pitched(v3, 12, 16)
    assert got is not None and got.shape == (12, 16) and got.data_ptr() == buf.data_ptr()
    assert mm._as_pitched(v3.reshape(-1, 10), 12, 16) is not None              # [12, 10] with row stride 16: still a view
    assert mm._as_pitched(buf[:, :10], 12, 16) is not None
    assert mm._as_pitched(buf[1:, :10], 11, 16) is None                        # not at the storage base
    assert mm._as_pitched(buf[:, :10].contiguous(), 12, 16) is None            # dense copy: pitch is V, not 16
    assert mm._as_pitched(buf.float()[:, :10], 12, 16) is None                 # wrong dtype
    assert mm._as_pitched(buf.view(3, 4, 16)[:, :2, :10], 6, 16) is None       # rows are not a plain enumeration


def test_grammar_lut_matches_tokenizer_tables():
    """decode.GrammarLUT (id ranges consumed by the fused sampler) == midi_tokenizer.py:517-535 as restated in
    tokenizer_tables: step 0 = eos + event ids, step i = the i-th parameter's contiguous id range."""
    from midi_b200.decode import GrammarLUT
    from midi_b200.tokenizer_tables import TokenizerTables
    tok = TokenizerTables("v2")
    g = GrammarLUT(tok, "cpu")
    assert (g.eos, g.pad, g.n_event_types) == (tok.eos_id, tok.pad_id, len(tok.event_ids))
    lut = g.lut.numpy()
    for name, params in tok.events.items():
        e = tok.event_ids[name] - (tok.eos_id + 1)
        for i, pn in enumerate(params):
            ids = tok.parameter_ids[pn]
            assert tuple(lut[e, i]) == (ids[0], ids[-1] + 1), (name, pn)
        assert (lut[e, len(params):] == 0).all()
        assert g.n_params[tok.event_ids[name]] == len(params)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the native one) prints ONE JSON line with the
    contract's keys and runs without a GPU."""
    import json
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train_tokens_per_sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bench_last_step_outputs(monkeypatch):
    """`bench.py --dump-outputs`: the loss and every trainable parameter with its gradient in float32, within the byte
    budget; a tensor over its share is sampled at the same seeded positions for parameter and gradient, run after run."""
    import importlib.util
    import midi_model as mm
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 1 << 20)
    torch.manual_seed(0)
    m = mm.MIDIModel(mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64))
    named = list(m.named_parameters())
    for _, p in named:
        p.grad = -2 * p.detach()
    out = bench.last_step_outputs(m, torch.tensor(1.5))
    assert set(out) == {"loss"} | {f"{k}.{n}" for n, _ in named for k in ("param", "grad")}
    assert out["loss"] == np.float32(1.5)
    assert all(a.dtype == np.float32 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= (1 << 20) + 4
    share = (1 << 20) // 4 // (2 * len(named))
    sampled = 0
    for n, p in named:
        a, g = out["param." + n], out["grad." + n]
        np.testing.assert_array_equal(g, -2 * a)
        full = p.detach().reshape(-1).numpy()
        if p.numel() <= share:
            np.testing.assert_array_equal(a, full)
        else:
            sampled += 1
            assert a.shape == (share,) and np.isin(a, full).all()
    assert sampled >= 3                                   # the two embedding tables and lm_head
    again = bench.last_step_outputs(m, torch.tensor(1.5))
    assert all(np.array_equal(out[k], again[k]) for k in out)


def test_no_cpu_fallback():
    import midi_model as mm
    from midi_b200.lib import B200Error
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64)
    m = mm.MIDIModel(cfg)
    with pytest.raises(B200Error):
        m.forward(torch.zeros(1, 2, 8, dtype=torch.long))
    with pytest.raises(B200Error):
        m.sample_top_p_k(torch.ones(1, 1, 3406) / 3406, 0.98, 20)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "midi-model_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), os.path.join(dp, f)


def test_synth_batch_is_grammar_valid():
    from midi_b200.synth import synth_batch
    from midi_b200.tokenizer_tables import TokenizerTables
    tok = TokenizerTables("v2")
    b = synth_batch(tok, 3, 50, seed=1, pad_tail=4)
    assert b.shape == (3, 50, 8) and b.dtype == torch.int64
    assert (b[:, 0, 0] == tok.bos_id).all() and (b[:, 0, 1:] == 0).all()
    assert (b[:, -4:] == 0).all()
    for row in b[:, 1:-4].reshape(-1, 8).tolist():
        assert tok.tokens2event(row) != []
    assert torch.equal(b, synth_batch(tok, 3, 50, seed=1, pad_tail=4))


def test_decode_descriptor_mirror_matches_the_header():
    """The ctypes mirror of b200_decode_desc (persistent generate kernel) has the size the C compiler gives the struct, and
    every field the header declares, in order."""
    import ctypes
    import re
    from midi_b200 import lib
    assert ctypes.sizeof(lib.DecodeDesc) == lib.query("b200_decode_desc_bytes")
    hdr = open(os.path.join(ROOT, "include", "midi_b200.h")).read()
    body = hdr[hdr.index("typedef struct b200_decode_desc {"):hdr.index("} b200_decode_desc;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for stmt in body.split("{", 1)[1].split(";"):
        stmt = stmt.strip()
        if not stmt:
            continue
        for part in stmt.split(","):
            names.append(re.findall(r"[A-Za-z_][A-Za-z_0-9]*", part)[-1])
    assert names == [f[0] for f in lib.DecodeDesc._fields_]


def test_generate_loop_modes():
    import midi_model as mm
    assert mm._loop_mode("persist") == "persist"
    assert mm._loop_mode("graph") is True and mm._loop_mode("nograph") is False and mm._loop_mode("eager") is False


def test_paged_kv_grow_keeps_cached_positions():
    """PagedKV.grow (contexts past max_position_embeddings: app.py's prompt + 4096 new events): after re-allocation every
    cached (row, head, position) is found through the new block table where it was before."""
    import torch
    from midi_b200.decode import PagedKV
    from midi_b200.engine import StackCfg
    cfg = StackCfg("net", 2, 4, 32, 64, 1e-6)          # 2 layers, 4 heads of 8
    kv = PagedKV(cfg, batch=3, capacity=20, page=8, device="cpu")
    assert kv.capacity == 24 and kv.max_pages == 3
    g = torch.Generator().manual_seed(0)
    for pools in (kv.k, kv.v):
        for li in range(cfg.n_layer):
            pools[li].copy_(torch.randn(pools[li].shape, generator=g).to(torch.bfloat16))

    def gather(pool, bt, page, b, h, t):
        return pool[int(bt[b, t // page]), h, t % page].clone()

    before = {(li, b, h, t): (gather(kv.k[li], kv.block_table, 8, b, h, t), gather(kv.v[li], kv.block_table, 8, b, h, t))
              for li in range(2) for b in range(3) for h in range(4) for t in (0, 7, 8, 19)}
    kv.length = 20
    kv.grow(25)
    assert kv.capacity >= 48 and kv.capacity % 8 == 0 and kv.block_table.shape == (3, kv.max_pages) and kv.length == 20
    for (li, b, h, t), (k0, v0) in before.items():
        assert torch.equal(gather(kv.k[li], kv.block_table, 8, b, h, t), k0)
        assert torch.equal(gather(kv.v[li], kv.block_table, 8, b, h, t), v0)
    kv.grow(10)                                          # no-op
    assert kv.capacity >= 48


def test_header_is_plain_c_and_a_c_program_can_bind_it(tmp_path):
    """include/midi_b200.h compiles stand-alone as C99 and as C++ (no CUDA headers), and a plain-C host program
    (tests/abi/abi_host.c) links libmidi_b200.so and exercises the entry points that need no GPU: version / size queries and
    the argument validation (error code + message) that precedes every launch."""
    import shutil
    import subprocess
    lib = _built()
    hdr = os.path.join(ROOT, "include", "midi_b200.h")
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-x", "c", hdr])
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Werror", "-fsyntax-only", "-x", "c++", hdr])
    exe = str(tmp_path / "abi_host")
    libdir = os.path.dirname(lib.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "abi", "abi_host.c"), "-L", libdir, "-lmidi_b200",
                           f"-Wl,-rpath,{libdir}", "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0 and "abi host ok" in r.stdout, r.stdout + r.stderr


def test_gemm_planner_reproduces_the_committed_sweep():
    """The tile / split-K planner (b200_gemm_plan: a host-side cost model, needs no GPU) still makes the choices that
    profiles/r2_gemm_plan_sweep.txt measured on a B200 for the 24 GEMM shapes of the benchmark step -- a change to the cost
    model has to come with a new sweep."""
    lib = _built()
    L = lib.load()
    n = 0
    for line in open(os.path.join(ROOT, "profiles", "r2_gemm_plan_sweep.txt")):
        m = re.match(r"(fwd|dgrad|wgrad)\s+rows=\s*(\d+) out=\s*(\d+) in=\s*(\d+) x\s*\d+ planner \((\d+), (\d+)\)", line)
        if not m:
            continue
        kind = m.group(1)
        R, O, I, bn, sp = map(int, m.groups()[1:])
        M, N, K, allow = {"fwd": (R, O, I, 0), "dgrad": (R, I, O, 0), "wgrad": (O, I, R, 1)}[kind]
        b, s = ctypes.c_int(0), ctypes.c_int(0)
        assert L.b200_gemm_plan(M, N, K, allow, ctypes.byref(b), ctypes.byref(s)) == 0
        assert (b.value, s.value) == (bn, sp), (kind, R, O, I, (bn, sp), (b.value, s.value))
        n += 1
    assert n == 24
    # shapes the LoRA adapters add (rank 64): skinny outputs take the 128-wide tile; the long-K gradient GEMMs split
    for M, N, K, allow, want_bn in ((131072, 64, 1024, 0, 128), (1024, 64, 131072, 1, 128), (64, 1024, 16384, 1, 128)):
        b, s = ctypes.c_int(0), ctypes.c_int(0)
        assert L.b200_gemm_plan(M, N, K, allow, ctypes.byref(b), ctypes.byref(s)) == 0
        assert b.value == want_bn and (s.value > 1) == bool(allow)
