"""The oracle (oracle/vv_oracle.py) against golden vectors produced by the reference's own modules
(oracle/make_golden.py).  CPU only; this is what pins the checker every CUDA parity test relies on."""
import numpy as np
import pytest
import torch

from oracle import vv_oracle as O
from oracle.make_golden import frame_sample
from vibevoice_b200.configuration import preset_config
from vibevoice_b200.synth import synth_state_dict

SEED = 1234


def close(a, b, rtol=1e-5, atol=1e-6):
    torch.testing.assert_close(a.float(), b.float(), rtol=rtol, atol=atol)


@pytest.mark.parametrize("n", [5, 10, 20, 30])
def test_dpm_tables_match_reference_scheduler(golden, n):
    g = golden("scheduler")[n]
    tab = O.dpm_tables(n)
    assert np.array_equal(tab.timesteps, g["timesteps"].numpy())          # integer bookkeeping: bit-exact
    assert np.array_equal(tab.sigmas, g["sigmas"].numpy())                 # fp32 table: bit-exact
    assert tab.order[0] == 1 and tab.order[-1] == 1 and (tab.order[1:-1] == 2).all()
    z, x0p = g["z0"].clone(), None
    for i in range(n):
        z, x0p = O.dpm_step(tab, i, g["vs"][i], z, x0p)
        close(z, g["traj"][i], rtol=0, atol=0)                             # scalar-table form is bit-exact in fp32


@pytest.mark.parametrize("n", [5, 10, 30])
def test_sde_dpm_tables_match_reference_scheduler(golden, n):
    """`sde-dpmsolver++` (the Gradio demo's scheduler, demo/gradio_demo.py:141-146; dpm_solver.py:680-686, 785-793): scalar tables +
    explicit variance noise reproduce the reference scheduler's trajectory bit for bit."""
    g = golden("scheduler")["sde%d" % n]
    tab = O.dpm_tables(n, algorithm_type="sde-dpmsolver++")
    assert np.array_equal(tab.timesteps, g["timesteps"].numpy())
    assert np.array_equal(tab.sigmas, g["sigmas"].numpy())
    z, x0p = g["z0"].clone(), None
    for i in range(n):
        z, x0p = O.dpm_step(tab, i, g["vs"][i], z, x0p, noise=g["noise"][i])
        close(z, g["traj"][i], rtol=0, atol=0)


def test_known_timesteps():
    # SURVEY 8a-4: N=10 -> 999,899,...,100 ; N=30 -> 999,966,932,...,33
    assert O.dpm_tables(10).timesteps.tolist() == [999, 899, 799, 699, 599, 500, 400, 300, 200, 100]
    t30 = O.dpm_tables(30).timesteps
    assert t30[0] == 999 and t30[1] == 966 and t30[2] == 932 and t30[-1] == 33
    assert abs(O.dpm_tables(10).sigmas[0] - 20291.3) < 1.0 and O.dpm_tables(10).sigmas[-1] == 0.0


def test_head_forward_and_sampler(golden):
    g = golden("head")
    cfg = preset_config(g["preset"])
    w = synth_state_dict(cfg, SEED, torch.float32, parts=("head",))
    y = O.head_forward(w, g["noisy"], g["t"], g["cond"])
    close(y, g["y"], rtol=1e-5, atol=1e-6)
    for n_steps, s in g["samples"].items():
        lat = O.sample_speech_tokens(w, s["pos"], s["neg"], s["cfg_scale"], n_steps, s["noise"])
        close(lat, s["latent"], rtol=1e-4, atol=2e-5)


def test_streaming_codec(golden):
    g = golden("codec")
    cfg = preset_config(g["preset"])
    w = synth_state_dict(cfg, SEED, torch.float32, parts=("acoustic_decoder", "acoustic_encoder", "semantic"))
    a, s = O.StreamState(g["n_rows"]), O.StreamState(g["n_rows"])
    for f, fr in enumerate(g["frames"]):
        if f in g["zero_before"]:
            a.set_to_zero(g["zero_before"][f]); s.set_to_zero(g["zero_before"][f])
        audio = O.decoder_frame(w, cfg.acoustic_tokenizer_config, fr["latent"], a, fr["rows"])
        assert audio.shape == (len(fr["rows"]), 1, 3200)
        close(audio, fr["audio"], rtol=1e-4, atol=1e-5)
        sem = O.encoder_frame(w, cfg.semantic_tokenizer_config, fr["audio"], s, fr["rows"])
        assert sem.shape == (len(fr["rows"]), 1, 128)
        close(sem, fr["semantic"], rtol=1e-4, atol=1e-5)
    enc = O.encoder_full(w, cfg.acoustic_tokenizer_config, g["wav"], "model.acoustic_tokenizer.encoder")
    close(enc, g["acoustic_encode_mean"], rtol=1e-4, atol=1e-5)
    sem = O.encoder_full(w, cfg.semantic_tokenizer_config, g["wav"], "model.semantic_tokenizer.encoder")
    close(sem, g["semantic_encode_full"], rtol=1e-4, atol=1e-5)


def test_connectors(golden):
    g = golden("connector")
    cfg = preset_config(g["preset"])
    w = synth_state_dict(cfg, SEED, torch.float32, parts=("connectors",))
    for name in ("acoustic", "semantic"):
        close(O.connector(w, f"model.{name}_connector", g[name]["x"]), g[name]["y"], rtol=1e-5, atol=1e-6)


def test_qwen2_prefill_and_decode(golden):
    g = golden("lm")
    cfg = preset_config(g["preset"])
    dc = cfg.decoder_config
    w = synth_state_dict(cfg, SEED, torch.float32, parts=("lm",))
    cache = O.KVCache(dc.num_hidden_layers)
    e = w["model.language_model.embed_tokens.weight"][g["ids"][0]]
    hs = O.qwen2_forward(w, dc, e, cache, 0)
    close(hs, g["hidden"][0], rtol=1e-4, atol=1e-5)
    for i, emb in enumerate(g["step_embeds"]):
        hs = O.qwen2_forward(w, dc, emb[0], cache, len(cache))
        close(hs, g["hidden"][i + 1], rtol=1e-4, atol=1e-5)
    assert len(cache) == g["ids"].shape[1] + len(g["step_embeds"])


def test_voice_prompt_embeds(golden):
    """a-9: acoustic encoder + Gaussian sampling + connector against the reference's `_process_speech_inputs` (same CPU RNG stream)."""
    g = golden("voice_prompt")
    cfg = preset_config(g["preset"])
    w = synth_state_dict(cfg, SEED, torch.float32, parts=("acoustic_encoder", "connectors"))
    torch.manual_seed(g["seed"])
    got = O.voice_prompt_embeds(w, cfg, g["wavs"], g["masks"])
    assert got.shape == g["connected"].shape == (7, cfg.decoder_config.hidden_size)
    close(got, g["connected"], rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("case", ["scripted", "free", "maxlen", "norefresh", "quirk", "voice", "sampled", "norefresh1", "sde"])
def test_generate_loop_matches_the_reference_generate(golden, case):
    """The whole loop (a-1 token state machine, a-2 negative CFG stream, a-8 state zeroing) against the reference's OWN
    `generate()` (modeling_vibevoice_inference.py:326-695) run on the same synthetic checkpoint by `oracle/make_golden.py::gen_loop`
    (loop body unmodified; transformers-4.51.3 glue restated in `oracle/ref_shim.py::install_generate_compat`).
    Token sequences and reach_max flags: exact.  Waveforms: fp32 on both sides, 1e-5."""
    from vibevoice_b200.synth import SynthTokenizer
    g = golden("loop")
    c = g[case]
    cfg = preset_config(g["preset"])
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    sd = synth_state_dict(cfg, SEED, torch.float32)
    torch.manual_seed(c["seed"])
    speech_embeds = None
    if "wavs" in c:                     # a-9: the prefill draws its Gaussian sample first, from the same CPU stream as the frame noise
        connected = O.voice_prompt_embeds(sd, cfg, c["wavs"], c["voice_masks"])
        speech_embeds, o = [], 0
        for b in range(c["ids"].shape[0]):
            m = c["speech_input_mask"][b][c["mask"][b].bool()]
            speech_embeds.append((m, connected[o:o + int(m.sum())]))
            o += int(m.sum())
    out = O.generate(sd, cfg, c["ids"], c["mask"], tok, cfg_scale=g["cfg_scale"], num_steps=g["num_steps"],
                     max_new_tokens=c["max_new_tokens"], max_length_times=c["max_length_times"], forced_tokens=c["scripts"],
                     refresh_negative=c["refresh_negative"], speech_embeds=speech_embeds, do_sample=c["do_sample"],
                     algorithm_type=c.get("algorithm_type", "dpmsolver++"))
    assert torch.equal(out.sequences, c["sequences"])
    assert torch.equal(out.reach_max_step_sample, c["reach_max"])
    assert len(out.speech_outputs) == len(c["audio"])
    for a, b in zip(out.speech_outputs, c["audio"]):
        assert (a is None) == (b is None)
        if a is not None:
            a = frame_sample(a)             # the fixture keeps a fixed half of every frame
            assert a.shape == b.shape
            rel = float((a.double() - b.double()).norm() / b.double().norm())
            assert rel < 1e-5, rel


def test_logical_negative_bookkeeping_is_the_reference_on_well_formed_sequences(golden):
    """The CUDA path keeps the negative stream by the rule the reference's mask/cache shifting implements -- "a row that is not in
    diffusion mode does not keep its new KV entry" (`vv_kv_commit` advance 0).  That rule (oracle `negative_bookkeeping="logical"`)
    is bit-identical to the reference-faithful bookkeeping on well-formed sequences, and differs on the one ill-formed pattern
    where the reference's two guards disagree (:603 vs :613) -- a stated deviation of the product path (DESIGN section 4)."""
    from vibevoice_b200.synth import SynthTokenizer
    g = golden("loop")
    cfg = preset_config(g["preset"])
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    sd = synth_state_dict(cfg, SEED, torch.float32)

    def run(c, mode):
        torch.manual_seed(c["seed"])
        return O.generate(sd, cfg, c["ids"], c["mask"], tok, cfg_scale=g["cfg_scale"], num_steps=g["num_steps"],
                          max_new_tokens=c["max_new_tokens"], max_length_times=c["max_length_times"], forced_tokens=c["scripts"],
                          negative_bookkeeping=mode)
    for case in ("scripted", "maxlen"):
        a, b = run(g[case], "reference"), run(g[case], "logical")
        assert torch.equal(a.sequences, b.sequences)
        for x, y in zip(a.speech_outputs, b.speech_outputs):
            assert torch.equal(x, y)
    a, b = run(g["quirk"], "reference"), run(g["quirk"], "logical")
    rel = float((a.speech_outputs[0] - b.speech_outputs[0]).norm() / a.speech_outputs[0].norm())
    assert rel > 1e-3                                    # the d,e,d row hears a different negative context ...
    assert torch.equal(a.speech_outputs[1], b.speech_outputs[1])      # ... the well-formed row does not


@pytest.mark.parametrize("case", ["eos", "windows", "short"])
def test_streaming_generate_matches_the_reference(golden, case):
    """SURVEY 8f-1 groundwork: the streaming-0.5B loop (split LM, type embeddings, EOS classifier, 5-token text windows / 6-frame
    speech windows) restated in `oracle/vv_streaming.py` against the reference's own streaming generate()
    (modeling_vibevoice_streaming_inference.py:412-725) on a synthetic split checkpoint.  Sequences and the max-length flag exact,
    waveform 1e-5."""
    from oracle import vv_streaming as VS
    g = golden("streaming")
    c = g[case]
    cfg = preset_config(g["preset"])
    sd = VS.streaming_state_dict(synth_state_dict(cfg, SEED, torch.float32), cfg, g["tts_layers"], eos_bias=c["eos_bias"])
    torch.manual_seed(c["seed"])
    out = VS.generate_streaming(sd, cfg, g["tts_layers"], c["prompt"], c["text"], g["neg_id"], cfg_scale=c["cfg_scale"],
                                num_steps=g["num_steps"], max_new_tokens=c["max_new_tokens"])
    assert torch.equal(out.sequences, c["sequences"])
    assert torch.equal(out.reach_max_step_sample, c["reach_max"])
    a, b = out.speech_outputs[0], c["audio"]
    assert (a is None) == (b is None)
    if a is not None:
        assert a.shape == b.shape
        assert float((a.double() - b.double()).norm() / b.double().norm()) < 1e-5
