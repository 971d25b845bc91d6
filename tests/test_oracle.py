"""Pin the CPU oracle (oracle/midi_oracle.py) against fixtures produced by the
unmodified reference (oracle/make_golden.py)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import midi_oracle as O
from midi_b200.tokenizer_tables import TokenizerTables

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")

TINY = O.ModelCfg(vocab=3406, n_layer=4, n_head=4, n_embd=32, n_inner=64)


def tiny_sd(g, dtype=torch.float32):
    return {k[3:]: torch.from_numpy(v).to(dtype) for k, v in g.items() if k.startswith("sd/")}


def test_tokenizer_tables_v2():
    t = TokenizerTables("v2")
    assert t.vocab_size == 3406 and t.max_token_seq == 8
    assert (t.pad_id, t.bos_id, t.eos_id) == (0, 1, 2)
    assert t.event_ids == {"note": 3, "patch_change": 4, "control_change": 5, "set_tempo": 6,
                           "time_signature": 7, "key_signature": 8}
    r = {k: (v[0], v[-1] + 1) for k, v in t.parameter_ids.items()}
    assert r["time1"] == (9, 137) and r["duration"] == (153, 2201) and r["mi"] == (3404, 3406)
    assert r["bpm"] == (2985, 3369) and r["pitch"] == (2345, 2473)
    ev = ["note", 3, 2, 1, 0, 60, 80, 4]
    toks = t.event2tokens(ev)
    assert len(toks) == 8 and t.tokens2event(toks) == ev
    assert TokenizerTables("v1").vocab_size == 3239


def test_tokenizer_tables_match_reference():
    """The id tables equal the reference tokenizer's (tests/golden/tokenizer.json, written by oracle/make_golden.py)."""
    with open(os.path.join(GOLDEN, "tokenizer.json")) as f:
        ref = json.load(f)
    for ver in ("v1", "v2"):
        a, b = TokenizerTables(ver), ref[ver]
        for attr in ("vocab_size", "pad_id", "bos_id", "eos_id", "events", "event_parameters", "event_ids",
                     "parameter_ids", "max_token_seq"):
            assert getattr(a, attr) == b[attr], attr
        assert a.id_events == {i: e for i, e in b["id_events"]}
        assert a.to_dict() == b["to_dict"]


def test_forward_fp32_golden(golden_tiny):
    g = golden_tiny
    sd = tiny_sd(g)
    batch = torch.from_numpy(g["batch"])
    x, y = batch[:, :-1], batch[:, 1:]
    hidden = O.forward(sd, TINY, x)
    np.testing.assert_allclose(hidden.reshape(-1, 32).numpy(), g["fp32/hidden"], rtol=2e-4, atol=2e-5)
    logits = O.forward_token(sd, TINY, hidden.reshape(-1, 32), y.reshape(-1, 8)[:, :-1])
    np.testing.assert_allclose(logits.numpy(), g["fp32/logits"], rtol=2e-4, atol=2e-5)
    loss = O.train_loss(sd, TINY, batch)
    assert abs(loss.item() - float(g["fp32/loss"])) < 1e-5
    rb = torch.from_numpy(g["rand_batch"])
    assert abs(O.train_loss(sd, TINY, rb).item() - float(g["fp32/rand_loss"])) < 1e-5


def test_grads_fp32_golden(golden_tiny):
    g = golden_tiny
    sd = {k: v.requires_grad_(True) for k, v in tiny_sd(g).items()}
    loss = O.train_loss(sd, TINY, torch.from_numpy(g["batch"]))
    loss.backward()
    for k, v in sd.items():
        gr = v.grad
        assert abs(gr.double().norm().item() - float(g["gradnorm/" + k])) <= 2e-4 * float(g["gradnorm/" + k]) + 1e-9, k
        ref = g["grad/" + k]
        np.testing.assert_allclose(gr[: ref.shape[0]].numpy(), ref, rtol=1e-3, atol=2e-6, err_msg=k)
    # padding_idx rows receive zero gradient in the reference (hf nn.Embedding(padding_idx=pad_token_id))
    assert np.all(g["grad/net.embed_tokens.weight"][0] == 0)
    assert np.all(g["grad/net_token.embed_tokens.weight"][0] == 0)


def test_forward_bf16_golden(golden_tiny):
    """bf16: same rounding points => close to the reference's own bf16 run (CPU kernels are
    deterministic, so this is tight), and the RoPE inv_freq buffer is the bf16-rounded one."""
    g = golden_tiny
    sd = tiny_sd(g, torch.bfloat16)
    batch = torch.from_numpy(g["batch"])
    x, y = batch[:, :-1], batch[:, 1:]
    ifn = O.default_inv_freq(8).to(torch.bfloat16)
    ift = O.default_inv_freq(32).to(torch.bfloat16)
    np.testing.assert_array_equal(ifn.float().numpy(), g["bf16/inv_freq_net"])
    np.testing.assert_array_equal(ift.float().numpy(), g["bf16/inv_freq_tok"])
    hidden = O.forward(sd, TINY, x)
    assert O.rel_fro(hidden.reshape(-1, 32).float(), torch.from_numpy(g["bf16/hidden"])) < 1.5e-2
    logits = O.forward_token(sd, TINY, hidden.reshape(-1, 32), y.reshape(-1, 8)[:, :-1])
    assert O.rel_fro(logits.float(), torch.from_numpy(g["bf16/logits"])) < 1.5e-2


def test_cached_forward_golden(golden_tiny):
    g = golden_tiny
    sd = tiny_sd(g)
    batch = torch.from_numpy(g["batch"])
    c = O.KV()
    hs = [O.forward(sd, TINY, batch[:, :5], c), O.forward(sd, TINY, batch[:, 5:6], c),
          O.forward(sd, TINY, batch[:, 6:9], c)]
    np.testing.assert_allclose(torch.cat(hs, 1).numpy(), g["fp32/cached_hidden"], rtol=2e-4, atol=2e-5)
    # and equals the uncached forward over the same 9 events
    full = O.forward(sd, TINY, batch[:, :9])
    np.testing.assert_allclose(torch.cat(hs, 1).numpy(), full.numpy(), rtol=2e-4, atol=2e-5)


def test_generate_greedy_golden(golden_tiny):
    g = golden_tiny
    sd = tiny_sd(g)
    tok = TokenizerTables("v2")
    ids = O.generate(sd, TINY, tok, None, batch_size=2, max_len=12, top_k=1,
                     generator=torch.Generator().manual_seed(0))
    np.testing.assert_array_equal(ids, g["gen/greedy_ids"])
    ids2 = O.generate(sd, TINY, tok, g["gen/prompt"], batch_size=2, max_len=10, top_k=1,
                      generator=torch.Generator().manual_seed(0))
    np.testing.assert_array_equal(ids2, g["gen/greedy_prompt_ids"])


def _app_stream_kwargs(name, g):
    from oracle.make_golden import APP_CASES
    kw = dict(APP_CASES[name])
    prompt = g["prompt"] if kw.pop("prompt", None) == "batch4" else None
    seed = kw.pop("seed", 0)
    tok = TokenizerTables("v2")
    deny = O.deny_ids(tok, kw.pop("disable_patch_change", False), kw.pop("disable_control_change", False),
                      kw.pop("disable_channels", None))
    return tok, prompt, seed, deny, kw


@pytest.mark.parametrize("case", ["greedy", "sampled", "plain"])
def test_app_stream_golden(golden_tiny, case):
    """oracle.generate_stream (+ deny masks, 4096-event window) == the events the reference's app.py generate() yields
    (tests/golden/app_stream.npz, produced by oracle/make_golden.py from the reference file itself)."""
    g = np.load(os.path.join(GOLDEN, "app_stream.npz"))
    tok, prompt, seed, deny, kw = _app_stream_kwargs(case, g)
    sd = tiny_sd(golden_tiny)
    blocks = list(O.generate_stream(sd, TINY, tok, prompt, generator=torch.Generator().manual_seed(seed), deny=deny,
                                    max_context=4096, **kw))
    P = blocks[0].shape[1]
    assert P == (1 if prompt is None else prompt.shape[1])
    evs = np.stack([b.numpy() for b in blocks[1:]], axis=1)
    np.testing.assert_array_equal(evs, g[case])
    assert not np.isin(evs, sorted(deny)).any()
    if case == "plain":      # no options: identical to MIDIModel.generate's continuation (midi_model.py:167-250)
        np.testing.assert_array_equal(evs, golden_tiny["gen/greedy_prompt_ids"][:, P:])


def test_app_stream_vs_live_reference(golden_tiny):
    """Three sampled rows with temperature, top-p / top-k, no patch changes and two channels denied == the events
    app.py's generate() yielded for the same call (the "options" case of tests/golden/app_stream.npz)."""
    g = np.load(os.path.join(GOLDEN, "app_stream.npz"))
    tok, prompt, seed, deny, kw = _app_stream_kwargs("options", g)
    assert prompt is None and deny == O.deny_ids(tok, True, False, [0, 3])
    blocks = list(O.generate_stream(tiny_sd(golden_tiny), TINY, tok, None, generator=torch.Generator().manual_seed(seed),
                                    deny=deny, max_context=4096, **kw))
    np.testing.assert_array_equal(np.stack([b.numpy() for b in blocks[1:]], axis=1), g["options"])


def test_sampler_golden(golden_tiny):
    g = golden_tiny
    probs = torch.from_numpy(g["samp/probs"])
    for name in "abcd":
        p, k = g[f"samp/{name}_pk"]
        s = O.sample_top_p_k(probs.clone(), float(p), int(k), generator=torch.Generator().manual_seed(5), stable=False)
        np.testing.assert_array_equal(s.numpy(), g[f"samp/{name}"])


def test_oracle_vs_live_reference_medium_shape():
    """Cross-check at tv2o-medium width with the compute kept small (4 layers, a (1, 9, 8) batch) against the reference's
    own class on the same seed-1 weights, which the drop-in class regenerates bit for bit (tests/golden/medium_4layer.npz:
    hidden states in full, logits as a seeded column sample plus the norm of all of them)."""
    import midi_model as mm
    from midi_b200.synth import synth_batch
    g = np.load(os.path.join(GOLDEN, "medium_4layer.npz"))
    torch.manual_seed(1)
    cfg = mm.MIDIModelConfig.get_config("v2", True, n_layer=4, n_head=16, n_embd=1024, n_inner=4096)
    model = mm.MIDIModel(cfg).eval()
    batch = synth_batch(model.tokenizer, 1, 9, seed=5)
    np.testing.assert_array_equal(batch.numpy(), g["batch"])
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    ocfg = O.cfg_from_hf(cfg)
    with torch.no_grad():
        h = O.forward(sd, ocfg, batch[:, :-1])
        l = O.forward_token(sd, ocfg, h.reshape(-1, 1024), batch[:, 1:].reshape(-1, 8)[:, :-1])
    assert O.rel_fro(h, torch.from_numpy(g["fp32/hidden"])) < 1e-5
    assert O.rel_fro(l[..., torch.from_numpy(g["logit_cols"])], torch.from_numpy(g["fp32/logits_sample"])) < 1e-5
    assert abs(l.double().norm().item() - float(g["fp32/logits_norm"])) < 1e-5 * float(g["fp32/logits_norm"])
