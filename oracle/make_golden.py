"""Generate tests/golden/*.npz from the UNMODIFIED reference -- run in the build
container only (`/root/reference` present):  python oracle/make_golden.py

The reference ships no tests or golden vectors (SURVEY.md section 4), so these fixtures
are outputs of the reference itself (torch 2.11.0 / transformers 5.5.0, CPU),
imported read-only through oracle/ref_loader.py.

  tiny.npz    tiny config (4L/4h/32/64 -> inner 1L/1h/32/16), seed-0 weights
              COMMITTED, inputs, fp32 + bf16 hidden / logits / loss, fp32 grads
              checksums, greedy generate ids, sample_top_p_k cases.
  medium.npz  tv2o-medium seed-0 init checksums + fp32 hidden/logits slices and
              loss on a (1,17,8) synthetic batch (weights regenerated from seed).
  app_stream.npz  events yielded by the reference's app.py generate() (app.py:27-120, executed from the reference
              file at run time, nothing copied) on the tiny model with the disable_* options, greedy and sampled.
  tokenizer.json  the reference tokenizer's id tables (v1 and v2): every attribute the drop-in mirrors, and to_dict().
  medium_4layer.npz  the reference's fp32 hidden states (full) and logits (a seeded sample of 256 vocabulary columns,
              plus the norm of all of them) for a 4-layer model of tv2o-medium width, seed-1 weights, on a (1, 9, 8) batch.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "midi-model_b200"))

from oracle import ref_loader  # noqa: E402
from midi_b200.synth import synth_batch, random_ids  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def ref_train_loss(model, batch):
    """train.py:168-185 with sample_seq=False, restated on the reference model object."""
    x = batch[:, :-1].contiguous()
    y = batch[:, 1:].contiguous()
    hidden = model.forward(x)
    hidden = hidden.reshape(-1, hidden.shape[-1])
    y = y.reshape(-1, y.shape[-1])
    xin = y[:, :-1]
    logits = model.forward_token(hidden, xin)
    loss = F.cross_entropy(logits.view(-1, model.tokenizer.vocab_size), y.view(-1), reduction="mean",
                           ignore_index=model.tokenizer.pad_id)
    return hidden, logits, loss


def tiny():
    mm, _ = ref_loader.load()
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64)
    model = mm.MIDIModel(cfg).eval()
    tok = model.tokenizer
    out = {}
    for k, v in model.state_dict().items():
        out["sd/" + k] = v.detach().numpy().astype(np.float32)
    batch = synth_batch(tok, 2, 13, seed=7, pad_tail=2)
    out["batch"] = batch.numpy()
    hidden, logits, loss = ref_train_loss(model, batch)
    loss.backward()
    out["fp32/hidden"] = hidden.detach().numpy()
    out["fp32/logits"] = logits.detach().numpy()
    out["fp32/loss"] = np.float32(loss.item())
    for k, p in model.named_parameters():
        g = p.grad.detach()
        out["gradnorm/" + k] = np.float64(g.double().norm().item())
        # big (vocab-sized) tensors: first 160 rows only; everything else in full
        out["grad/" + k] = (g[:160] if g.shape[0] > 1000 else g).numpy().astype(np.float32)
    # uniform random ids (kernel-parity variant)
    rb = random_ids(tok.vocab_size, 2, 9, seed=3)
    out["rand_batch"] = rb.numpy()
    with torch.no_grad():
        h2, l2, loss2 = ref_train_loss(model, rb)
    out["fp32/rand_hidden"] = h2.numpy()
    out["fp32/rand_loss"] = np.float32(loss2.item())
    # bf16 run of the reference itself (module cast rounds the RoPE inv_freq buffers)
    m16 = mm.MIDIModel(cfg)
    m16.load_state_dict(model.state_dict())
    m16 = m16.to(torch.bfloat16).eval()
    out["bf16/inv_freq_net"] = m16.net.rotary_emb.inv_freq.float().numpy()
    out["bf16/inv_freq_tok"] = m16.net_token.rotary_emb.inv_freq.float().numpy()
    with torch.no_grad():
        hb, lb, lossb = ref_train_loss(m16, batch)
    out["bf16/hidden"] = hb.float().numpy()
    out["bf16/logits"] = lb.float().numpy()
    out["bf16/loss"] = np.float32(lossb.float().item())
    # KV-cached incremental forward == full forward (public forward(x, cache) API)
    from transformers import DynamicCache
    with torch.no_grad():
        c = DynamicCache()
        h_a = model.forward(batch[:, :5], cache=c)
        h_b = model.forward(batch[:, 5:6], cache=c)
        h_c = model.forward(batch[:, 6:9], cache=c)       # q_len>1 with past
    out["fp32/cached_hidden"] = torch.cat([h_a, h_b, h_c], dim=1).numpy()
    # greedy generate (top_k=1), free running
    ids = model.generate(prompt=None, batch_size=2, max_len=12, top_k=1, generator=torch.Generator().manual_seed(0))
    out["gen/greedy_ids"] = ids
    prompt = batch[:, :4].numpy()
    ids2 = model.generate(prompt=prompt, batch_size=2, max_len=10, top_k=1, generator=torch.Generator().manual_seed(0))
    out["gen/prompt"] = prompt
    out["gen/greedy_prompt_ids"] = ids2
    # sampler cases (CPU generator -> deterministic draws)
    g = torch.Generator().manual_seed(11)
    logits_s = torch.randn(4, 1, tok.vocab_size, generator=g) * 3.0
    mask = torch.zeros(4, 1, tok.vocab_size, dtype=torch.int64)
    mask[..., 9:137] = 1
    probs = torch.softmax(logits_s, dim=-1) * mask
    out["samp/probs"] = probs.numpy()
    for name, (p, k) in {"a": (0.98, 20), "b": (0.5, 5), "c": (1.0, 1), "d": (0.9, 3406)}.items():
        gg = torch.Generator().manual_seed(5)
        s = model.sample_top_p_k(probs.clone(), p, k, generator=gg)
        out[f"samp/{name}"] = s.numpy()
        out[f"samp/{name}_pk"] = np.array([p, k], dtype=np.float64)
    np.savez_compressed(os.path.join(OUT, "tiny.npz"), **out)
    print("tiny.npz:", len(out), "arrays, loss", float(loss), "bf16 loss", float(lossb))


def medium():
    mm, _ = ref_loader.load()
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.from_name("tv2o-medium")
    model = mm.MIDIModel(cfg).eval()
    tok = model.tokenizer
    out = {}
    sd = model.state_dict()
    out["n_tensors"] = np.int64(len(sd))
    out["n_params"] = np.int64(sum(v.numel() for v in sd.values()))
    for k in ["net.embed_tokens.weight", "net.layers.0.self_attn.q_proj.weight", "net.layers.11.mlp.down_proj.weight",
              "net_token.layers.2.mlp.up_proj.weight", "net_token.embed_tokens.weight", "lm_head.weight",
              "net.norm.weight"]:
        v = sd[k].double()
        out["init/" + k] = np.array([v.sum().item(), v.abs().sum().item(), v.flatten()[12345 % v.numel()].item()])
    batch = synth_batch(tok, 1, 17, seed=1234)
    out["batch"] = batch.numpy()
    with torch.no_grad():
        hidden, logits, loss = ref_train_loss(model, batch)
    out["fp32/hidden"] = hidden.numpy()[:, :64]
    out["fp32/hidden_norm"] = np.float64(hidden.double().norm().item())
    out["fp32/logits"] = logits.numpy()[:, :, :128]
    out["fp32/logits_norm"] = np.float64(logits.double().norm().item())
    out["fp32/loss"] = np.float32(loss.item())
    np.savez_compressed(os.path.join(OUT, "medium.npz"), **out)
    print("medium.npz: loss", float(loss))


def ref_app_generate(model, tokenizer):
    """The reference's `generate` generator function of app.py:27-120, compiled from the reference file itself (the module
    cannot be imported: gradio / synthesizer dependencies) into a namespace holding its two globals."""
    import ast
    import tqdm
    from transformers import DynamicCache
    path = os.path.join(ref_loader.REF_DIR, "app.py")
    tree = ast.parse(open(path).read(), filename=path)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "generate"]
    assert len(fn) == 1
    ns = {"torch": torch, "np": np, "tqdm": tqdm, "F": F, "DynamicCache": DynamicCache, "model": model, "tokenizer": tokenizer}
    exec(compile(ast.Module(body=fn, type_ignores=[]), path, "exec"), ns)
    return ns["generate"]


APP_CASES = {
    "greedy": dict(prompt=None, batch_size=2, max_len=14, top_k=1, disable_patch_change=True, disable_control_change=True,
                   disable_channels=list(range(9))),
    "sampled": dict(prompt="batch4", batch_size=2, max_len=12, temp=1.0, top_p=0.98, top_k=20, disable_patch_change=False,
                    disable_control_change=True, disable_channels=[9], seed=3),
    "plain": dict(prompt="batch4", batch_size=2, max_len=10, top_k=1),
    "options": dict(prompt=None, batch_size=3, max_len=9, temp=0.9, top_p=0.95, top_k=10, disable_patch_change=True,
                    disable_control_change=False, disable_channels=[0, 3], seed=21),
}


def app_stream():
    mm, _ = ref_loader.load()
    torch.manual_seed(0)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=4, n_embd=32, n_inner=64)
    model = mm.MIDIModel(cfg).eval()                    # same seed-0 weights as tiny.npz
    gen = ref_app_generate(model, model.tokenizer)
    batch = synth_batch(model.tokenizer, 2, 13, seed=7, pad_tail=2)
    out = {"prompt": batch[:, :4].numpy()}
    for name, kw in APP_CASES.items():
        kw = dict(kw)
        if kw.get("prompt") == "batch4":
            kw["prompt"] = batch[:, :4].numpy()
        seed = kw.pop("seed", 0)
        evs = list(gen(generator=torch.Generator().manual_seed(seed), **kw))
        out[name] = np.stack(evs, axis=1)
        print("app_stream", name, out[name].shape)
    np.savez_compressed(os.path.join(OUT, "app_stream.npz"), **out)


TOKENIZER_ATTRS = ("vocab_size", "pad_id", "bos_id", "eos_id", "events", "event_parameters", "event_ids", "parameter_ids",
                   "max_token_seq")


def tokenizer():
    """id_events is stored as [id, name] pairs: JSON object keys are strings."""
    import json
    _, rt = ref_loader.load()
    out = {}
    for ver in ("v1", "v2"):
        t = rt.MIDITokenizer(ver)
        out[ver] = {a: getattr(t, a) for a in TOKENIZER_ATTRS}
        out[ver]["id_events"] = sorted([i, e] for i, e in t.id_events.items())
        out[ver]["to_dict"] = t.to_dict()
    with open(os.path.join(OUT, "tokenizer.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
        f.write("\n")


MEDIUM_4LAYER_COLS = 256


def medium_4layer():
    mm, _ = ref_loader.load()
    torch.manual_seed(1)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=16, n_embd=1024, n_inner=4096)
    model = mm.MIDIModel(cfg).eval()
    batch = synth_batch(model.tokenizer, 1, 9, seed=5)
    with torch.no_grad():
        h = model.forward(batch[:, :-1])
        lg = model.forward_token(h.reshape(-1, 1024), batch[:, 1:].reshape(-1, 8)[:, :-1])
    cols = np.sort(np.random.default_rng(0).choice(lg.shape[-1], MEDIUM_4LAYER_COLS, replace=False))
    out = {"batch": batch.numpy(), "fp32/hidden": h.numpy(), "logit_cols": cols, "fp32/logits_sample": lg.numpy()[..., cols],
           "fp32/logits_norm": np.float64(lg.double().norm().item())}
    np.savez_compressed(os.path.join(OUT, "medium_4layer.npz"), **out)
    print("medium_4layer.npz: hidden", tuple(h.shape), "logits", tuple(lg.shape))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(8)
    steps = {"tiny": tiny, "medium": medium, "app_stream": app_stream, "tokenizer": tokenizer, "medium_4layer": medium_4layer}
    for name in sys.argv[1:] or steps:
        steps[name]()
