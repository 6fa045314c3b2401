"""TEST INFRASTRUCTURE -- generates `tests/golden/*.pt` by running the UNMODIFIED reference modules
(imported from /root/reference through `oracle/ref_shim.py`) on seeded synthetic checkpoints.

    python -m oracle.make_golden [name ...]   # rewrites tests/golden/ (all fixtures, or the named ones)

The reference has no golden vectors of its own (SURVEY section 4); these fixtures are what pins the oracle
(`oracle/vv_oracle.py`) and, through it, the CUDA path.  Only runs in the build container (the GPU box
has no /root/reference); the fixtures it writes are committed.
"""
from __future__ import annotations

import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import ref_shim  # noqa: E402
from vibevoice_b200.configuration import preset_config  # noqa: E402
from vibevoice_b200.synth import SynthTokenizer, synth_state_dict  # noqa: E402

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
SEED = 1234
FRAME = 3200


def frame_sample(wav: torch.Tensor) -> torch.Tensor:
    """The part of a waveform `loop.pt` stores: the same fixed, seeded half of the samples of every 3200-sample frame (last axis).
    Keeps the fixture under 1 MB; the tests compare waveforms at these positions, so a length mismatch still fails."""
    keep = torch.randperm(FRAME, generator=torch.Generator().manual_seed(0))[:FRAME // 2].sort().values
    return wav.unflatten(-1, (-1, FRAME))[..., keep].flatten(-2)


def _sub(sd, prefix):
    return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}


def _ref_cfg(ns, cfg):
    """reference VibeVoiceConfig object built from our attribute bag (same JSON schema)."""
    d = cfg.to_dict()
    dec = dict(d["decoder_config"]); dec["model_type"] = "qwen2"; dec.pop("_attn_implementation", None)
    return ns.cfg.VibeVoiceConfig(acoustic_tokenizer_config=d["acoustic_tokenizer_config"],
                                  semantic_tokenizer_config=d["semantic_tokenizer_config"],
                                  decoder_config=dec, diffusion_head_config=d["diffusion_head_config"])


def gen_scheduler(ns):
    """Raw scheduler trajectories on a scripted model output (dpm_solver.py:321-423, 935-1022)."""
    out = {}
    for n in (5, 10, 20, 30):
        s = ns.dpm.DPMSolverMultistepScheduler(num_train_timesteps=1000, beta_schedule="cosine",
                                               prediction_type="v_prediction")
        s.set_timesteps(n)
        g = torch.Generator().manual_seed(100 + n)
        z = torch.randn(3, 64, generator=g)
        vs = torch.randn(n, 3, 64, generator=g)
        traj = []
        zz = z.clone()
        for i, t in enumerate(s.timesteps):
            zz = s.step(vs[i], t, zz).prev_sample
            traj.append(zz.clone())
        out[n] = dict(timesteps=s.timesteps.clone(), sigmas=s.sigmas.clone(), z0=z, vs=vs, traj=torch.stack(traj))
    # SDE variant as the Gradio demo configures it (demo/gradio_demo.py:141-146), variance noise passed explicitly
    for n in (5, 10, 30):
        base = ns.dpm.DPMSolverMultistepScheduler(num_train_timesteps=1000, beta_schedule="cosine", prediction_type="v_prediction")
        s = base.from_config(base.config, algorithm_type="sde-dpmsolver++", beta_schedule="squaredcos_cap_v2")
        s.set_timesteps(n)
        g = torch.Generator().manual_seed(200 + n)
        z = torch.randn(3, 64, generator=g)
        vs = torch.randn(n, 3, 64, generator=g)
        ns_ = torch.randn(n, 3, 64, generator=g)
        traj = []
        zz = z.clone()
        for i, t in enumerate(s.timesteps):
            zz = s.step(vs[i], t, zz, variance_noise=ns_[i]).prev_sample
            traj.append(zz.clone())
        out["sde%d" % n] = dict(timesteps=s.timesteps.clone(), sigmas=s.sigmas.clone(), z0=z, vs=vs, noise=ns_, traj=torch.stack(traj))
    return out


def gen_head(ns, preset="tiny"):
    cfg = preset_config(preset)
    rc = _ref_cfg(ns, cfg)
    sd = synth_state_dict(cfg, SEED, torch.float32, parts=("head",))
    head = ns.head.VibeVoiceDiffusionHead(rc.diffusion_head_config).eval()
    missing = head.load_state_dict(_sub(sd, "model.prediction_head."), strict=True)
    g = torch.Generator().manual_seed(7)
    H = cfg.decoder_config.hidden_size
    noisy, cond = torch.randn(6, 64, generator=g), torch.randn(6, H, generator=g)
    t = torch.tensor([999.0, 500.0, 33.0, 999.0, 500.0, 33.0])
    with torch.no_grad():
        y = head(noisy, t, condition=cond)
    # full CFG sampler through the reference's own method with a stand-in `self`
    infer = sys.modules["vibevoice.modular.modeling_vibevoice_inference"].VibeVoiceForConditionalGenerationInference
    samples = {}
    for n_steps, cfg_scale in ((5, 1.5), (10, 1.3), (30, 1.3)):
        sched = ns.dpm.DPMSolverMultistepScheduler(num_train_timesteps=1000, beta_schedule="cosine",
                                                   prediction_type="v_prediction")
        head.device  # noqa  (PreTrainedModel property used by :700)
        fake = types.SimpleNamespace(model=types.SimpleNamespace(noise_scheduler=sched, prediction_head=head),
                                     ddpm_inference_steps=n_steps, config=types.SimpleNamespace(acoustic_vae_dim=64))
        pos, neg = torch.randn(2, H, generator=g), torch.randn(2, H, generator=g)
        torch.manual_seed(11 + n_steps)
        noise = torch.randn(4, 64)
        torch.manual_seed(11 + n_steps)
        lat = infer.sample_speech_tokens(fake, pos, neg, cfg_scale=cfg_scale)
        samples[n_steps] = dict(pos=pos, neg=neg, cfg_scale=cfg_scale, noise=noise, latent=lat.clone())
    return dict(preset=preset, noisy=noisy, cond=cond, t=t, y=y, samples=samples)


def _tokenizer_models(ns, cfg):
    rc = _ref_cfg(ns, cfg)
    sd = synth_state_dict(cfg, SEED, torch.float32, parts=("acoustic_decoder", "acoustic_encoder", "semantic"))
    ac = ns.tok.VibeVoiceAcousticTokenizerModel(rc.acoustic_tokenizer_config).eval()
    ac.load_state_dict(_sub(sd, "model.acoustic_tokenizer."), strict=True)
    se = ns.tok.VibeVoiceSemanticTokenizerModel(rc.semantic_tokenizer_config).eval()
    se.load_state_dict(_sub(sd, "model.semantic_tokenizer."), strict=True)
    return ac, se


def gen_codec(ns, preset="tiny"):
    """Streaming decode/encode over several frames, ragged row subsets, and a `set_to_zero` (speech_end)."""
    cfg = preset_config(preset)
    ac, se = _tokenizer_models(ns, cfg)
    g = torch.Generator().manual_seed(21)
    n_rows = 3
    script = [[0, 1, 2], [0, 2], [0, 1, 2], [1], [0, 1, 2], [0, 1, 2]]   # rows decoding at each frame
    zero_before = {4: [0]}                                              # speech_end for row 0 before frame 4
    a_cache, s_cache = ns.tok.VibeVoiceTokenizerStreamingCache(), ns.tok.VibeVoiceTokenizerStreamingCache()
    frames = []
    with torch.no_grad():
        for f, rows in enumerate(script):
            if f in zero_before:
                zr = torch.tensor(zero_before[f])
                a_cache.set_to_zero(zr); s_cache.set_to_zero(zr)
            lat = torch.randn(len(rows), 1, 64, generator=g)
            idx = torch.tensor(rows)
            audio = ac.decode(lat, cache=a_cache, sample_indices=idx, use_cache=True)
            sem = se.encode(audio, cache=s_cache, sample_indices=idx, use_cache=True).mean
            frames.append(dict(rows=rows, latent=lat, audio=audio.clone(), semantic=sem.clone()))
        # non-streaming equivalents for one row (also what voice-prompt prefill uses for the encoder)
        wav = torch.randn(2, 1, 3200 * 3 + 777, generator=g) * 0.1
        enc_mean = ac.encode(wav).mean
        sem_full = se.encode(wav).mean
    return dict(preset=preset, n_rows=n_rows, zero_before=zero_before, frames=frames, wav=wav,
                acoustic_encode_mean=enc_mean, semantic_encode_full=sem_full)


def gen_connector(ns, preset="tiny"):
    cfg = preset_config(preset)
    sd = synth_state_dict(cfg, SEED, torch.float32, parts=("connectors",))
    H = cfg.decoder_config.hidden_size
    g = torch.Generator().manual_seed(31)
    out = {}
    for name, din in (("acoustic", 64), ("semantic", 128)):
        m = ns.modeling.SpeechConnector(din, H).eval()
        m.load_state_dict(_sub(sd, f"model.{name}_connector."), strict=True)
        x = torch.randn(3, 1, din, generator=g)
        with torch.no_grad():
            out[name] = dict(x=x, y=m(x))
    return dict(preset=preset, **out)


def build_ref_model(ns, cfg, dtype=torch.float32):
    """Full reference inference model with synthetic weights (used by the loop fixture)."""
    infer_mod = sys.modules["vibevoice.modular.modeling_vibevoice_inference"]
    rc = _ref_cfg(ns, cfg)
    rc.decoder_config._attn_implementation = "sdpa"
    model = infer_mod.VibeVoiceForConditionalGenerationInference(rc)
    sd = synth_state_dict(cfg, SEED, torch.float32)
    sd = {k: v for k, v in sd.items()}
    if cfg.decoder_config.tie_word_embeddings:
        sd["lm_head.weight"] = sd["model.language_model.embed_tokens.weight"]
    res = model.load_state_dict(sd, strict=False)
    bad = [k for k in res.missing_keys if "fix_std" not in k and "rotary" not in k]
    assert not bad and not res.unexpected_keys, (bad, res.unexpected_keys)
    return model.eval()


def gen_lm(ns, preset="tiny"):
    """Installed transformers Qwen2Model (the third-party arithmetic the reference calls at
    modeling_vibevoice.py:121): prefill + single-token decode steps."""
    from transformers import Qwen2Config, Qwen2Model
    cfg = preset_config(preset)
    dc = cfg.decoder_config
    qc = Qwen2Config(hidden_size=dc.hidden_size, intermediate_size=dc.intermediate_size,
                     num_hidden_layers=dc.num_hidden_layers, num_attention_heads=dc.num_attention_heads,
                     num_key_value_heads=dc.num_key_value_heads, head_dim=dc.head_dim,
                     max_position_embeddings=dc.max_position_embeddings, rms_norm_eps=dc.rms_norm_eps,
                     rope_theta=dc.rope_theta, vocab_size=dc.vocab_size, tie_word_embeddings=True,
                     attn_implementation="eager")
    m = Qwen2Model(qc).eval()
    sd = synth_state_dict(cfg, SEED, torch.float32, parts=("lm",))
    res = m.load_state_dict(_sub(sd, "model.language_model."), strict=False)
    assert not [k for k in res.missing_keys if "rotary" not in k] and not res.unexpected_keys, res
    g = torch.Generator().manual_seed(41)
    ids = torch.randint(0, dc.vocab_size - 20, (1, 9), generator=g)
    steps = torch.randn(3, 1, 1, dc.hidden_size, generator=g) * 0.05
    with torch.no_grad():
        o = m(input_ids=ids, use_cache=True)
        hs = [o.last_hidden_state[0].clone()]
        pkv = o.past_key_values
        for e in steps:
            o = m(inputs_embeds=e, past_key_values=pkv, use_cache=True)
            pkv = o.past_key_values
            hs.append(o.last_hidden_state[0].clone())
    return dict(preset=preset, ids=ids, step_embeds=steps, hidden=hs)


def gen_voice_prompt(ns, preset="tiny"):
    """The reference's own `_process_speech_inputs` (modeling_vibevoice_inference.py:149-163) on two ragged voice prompts."""
    cfg = preset_config(preset)
    ac, _ = _tokenizer_models(ns, cfg)
    sd = synth_state_dict(cfg, SEED, torch.float32, parts=("connectors",))
    con = ns.modeling.SpeechConnector(64, cfg.decoder_config.hidden_size).eval()
    con.load_state_dict(_sub(sd, "model.acoustic_connector."), strict=True)
    from vibevoice_b200.synth import SPEECH_BIAS_FACTOR, SPEECH_SCALING_FACTOR
    infer = sys.modules["vibevoice.modular.modeling_vibevoice_inference"].VibeVoiceForConditionalGenerationInference
    fake = types.SimpleNamespace(model=types.SimpleNamespace(acoustic_tokenizer=ac, acoustic_connector=con,
                                                             speech_bias_factor=torch.tensor(SPEECH_BIAS_FACTOR),
                                                             speech_scaling_factor=torch.tensor(SPEECH_SCALING_FACTOR)))
    g = torch.Generator().manual_seed(51)
    wavs = torch.zeros(2, 3200 * 3 + 100)
    wavs[0] = torch.randn(wavs.shape[1], generator=g) * 0.05
    wavs[1, :3200 * 2 + 7] = torch.randn(3200 * 2 + 7, generator=g) * 0.05
    masks = torch.zeros(2, 4, dtype=torch.bool)
    masks[0, :4] = True
    masks[1, :3] = True
    torch.manual_seed(77)
    feats, connected = infer._process_speech_inputs(fake, wavs, masks)
    return dict(preset=preset, wavs=wavs, masks=masks, seed=77, features=feats.clone(), connected=connected.clone())


def _scripted(tok, s):
    m = {"d": tok.speech_diffusion_id, "e": tok.speech_end_id, "s": tok.speech_start_id, "x": tok.eos_token_id}
    return [m[c] for c in s]


def gen_loop(ns, preset="tiny"):
    """The reference's own `generate()` (modeling_vibevoice_inference.py:326-695), loop body unmodified, on the synthetic tiny
    checkpoint; transformers-4.51.3 GenerationMixin glue restated by `ref_shim.install_generate_compat()`.  Three cases:
      scripted  B=2, ragged left-padded prompts, scripts with a speaker turn (<end>,<start>) and per-row EOS
                -> negative-stream restart, cache corrections for non-diffusing rows, codec-state zeroing, finished rows
      free      B=1, the constrained argmax itself drives the state machine
      maxlen    B=2 ragged, all-diffusion scripts, max_length_times=0.5 -> per-sample step limit / reach_max_step_sample
      norefresh B=2 ragged, two different speaker-turn scripts, refresh_negative=False
      streamed / stopped  B=2 with the reference AudioStreamer; with `stop_check_fn` firing after three steps
      sde       B=2 ragged scripted, scheduler replaced by sde-dpmsolver++
      norefresh1 B=1, two speaker turns, refresh_negative=False (no cache correction can occur: the product path supports this case)
      quirk     B=2 ragged, ill-formed d,e,d row: pins the reference's guard off-by-one in the cache correction
      sampled   B=2 ragged, do_sample=True
      voice     B=2 ragged, `is_prefill=True` with two voice prompts (acoustic encoder + Gaussian sample + connector, :149-163, 216-224)"""
    ref_shim.install_generate_compat()
    cfg = preset_config(preset)
    model = build_ref_model(ns, cfg)
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    V = cfg.decoder_config.vocab_size
    steps, cfg_scale = 5, 1.3
    model.set_ddpm_inference_steps(steps)

    def run(ids, mask, scripts, max_new_tokens, seed, max_length_times=2, refresh_negative=True, do_sample=False, streamer=False,
            stop_after_calls=None):
        ref_shim.script_tokens(ids.shape[1], scripts)
        torch.manual_seed(seed)
        extra = {}
        st = None
        if streamer:                                 # the reference's own AudioStreamer (vibevoice/modular/streamer.py:13-92)
            import importlib
            st = importlib.import_module("vibevoice.modular.streamer").AudioStreamer(batch_size=ids.shape[0])
            extra["audio_streamer"] = st
        if stop_after_calls is not None:
            calls = {"n": 0}

            def stop_fn():
                calls["n"] += 1
                return calls["n"] > stop_after_calls
            extra["stop_check_fn"] = stop_fn
        out = model.generate(**extra, input_ids=ids.clone(), attention_mask=mask.clone(), tokenizer=tok, cfg_scale=cfg_scale,
                             max_new_tokens=max_new_tokens, speech_tensors=None, speech_masks=None,
                             speech_input_mask=torch.zeros_like(ids, dtype=torch.bool), show_progress_bar=False, verbose=False,
                             is_prefill=False, max_length_times=max_length_times, refresh_negative=refresh_negative,
                             generation_config={"do_sample": True, "top_k": 0} if do_sample else None)
        ref_shim.script_tokens()
        audio = [None if a is None else frame_sample(a) for a in out.speech_outputs]
        streamed = None
        if st is not None:                           # queue contents per row, stop signal (None) included
            streamed = []
            for r, q in enumerate(st.audio_queues):
                items, o = [], 0
                while not q.empty():
                    it = q.get()
                    if it is not None:               # each chunk is the row's next frame: stored as a view of the row's waveform
                        n = frame_sample(it).shape[-1]
                        assert torch.equal(frame_sample(it), audio[r][..., o:o + n])
                        it, o = audio[r][..., o:o + n], o + n
                    items.append(it)
                streamed.append(items)
        return dict(streamed=streamed, stop_after_calls=stop_after_calls,
                    ids=ids, mask=mask, scripts=scripts, max_new_tokens=max_new_tokens, seed=seed, max_length_times=max_length_times, refresh_negative=refresh_negative, do_sample=do_sample,
                    sequences=out.sequences.clone(), reach_max=out.reach_max_step_sample.clone(), audio=audio)

    g = torch.Generator().manual_seed(3)
    L0 = 12
    ids = torch.randint(0, V - 20, (2, L0), generator=g)
    ids[:, -1] = tok.speech_start_id
    mask = torch.ones(2, L0, dtype=torch.long)
    mask[1, :4] = 0
    ids[1, :4] = tok.pad_token_id
    scripted = run(ids, mask, [_scripted(tok, "dddesddx"), _scripted(tok, "ddddddddx")], 40, 0)
    # free-running: the first prompt seed whose constrained argmax emits at least two diffusion tokens (random-init weights pick
    # <eos> or <speech_end> straight away for most prompts, which would leave the audio branch untested)
    free = None
    for pseed in range(64):
        gp = torch.Generator().manual_seed(100 + pseed)
        ids1 = torch.randint(0, V - 20, (1, 9), generator=gp)
        ids1[:, -1] = tok.speech_start_id
        cand = run(ids1, torch.ones_like(ids1), None, 8, 1)
        if int((cand["sequences"][0, 9:] == tok.speech_diffusion_id).sum()) >= 2:
            free = dict(cand, prompt_seed=100 + pseed)
            break
    assert free is not None, "no free-running prompt with diffusion tokens among 64 seeds"
    # per-sample step limit (:531-539): ragged rows have different max_step_per_sample under a small max_length_times
    maxlen = run(ids, mask, [_scripted(tok, "d"), _scripted(tok, "d")], 40, 2, max_length_times=0.5)
    # refresh_negative=False (:503-517): negative stream forwarded every step, never restarted, batch-coupled corrections
    norefresh = run(ids, mask, [_scripted(tok, "dddesddx"), _scripted(tok, "desdddddx")], 40, 3, refresh_negative=False)
    # audio_streamer hand-off (:443-447, :525-539, :653-655, :677-678: the loop ends as soon as ANY row's stream is finished) and the
    # cooperative stop hook (:434-440)
    streamed = run(ids, mask, [_scripted(tok, "dddesddx"), _scripted(tok, "ddddddddx")], 40, 8, streamer=True)
    stopped = run(ids, mask, [_scripted(tok, "d"), _scripted(tok, "d")], 40, 9, streamer=True, stop_after_calls=3)
    # sde-dpmsolver++ as the Gradio demo installs it (demo/gradio_demo.py:141-146); on the CPU every step's variance noise comes from the
    # global generator, interleaved with the per-frame draw
    ode_sched = model.model.noise_scheduler
    model.model.noise_scheduler = ode_sched.from_config(ode_sched.config, algorithm_type="sde-dpmsolver++", beta_schedule="squaredcos_cap_v2")
    model.set_ddpm_inference_steps(steps)
    sde = run(ids, mask, [_scripted(tok, "dddesddx"), _scripted(tok, "ddddddddx")], 40, 10)
    sde["algorithm_type"] = "sde-dpmsolver++"
    model.model.noise_scheduler = ode_sched
    model.set_ddpm_inference_steps(steps)
    g1 = torch.Generator().manual_seed(31)
    ids_one = torch.randint(0, V - 20, (1, 10), generator=g1)
    ids_one[:, -1] = tok.speech_start_id
    norefresh1 = run(ids_one, torch.ones_like(ids_one), [_scripted(tok, "ddesdddesdx")], 40, 7, refresh_negative=False)
    # ill-formed turn (<speech_end> followed directly by diffusion) while the other row diffuses: the off-by-one guard of the
    # correction block (:603 vs :613) hides slot correct_cnt instead of the newest entry (see vv_oracle.NegativeStream)
    quirk = run(ids, mask, [_scripted(tok, "dedddx"), _scripted(tok, "ddddddx")], 40, 4)
    # do_sample=True (:493-496): multinomial over the constrained scores on the global CPU generator, interleaved with the noise draws.
    # top_k=0: HF's default top_k=50 warper runs BEFORE the constraint processor and, with random-init weights, leaves none of the
    # valid ids finite (softmax of all -inf -> NaN inside the reference); temperature / top_p stay at their neutral defaults.
    sampled = run(ids, mask, None, 10, 6, do_sample=True)
    # voice-prompt prefill (a-9) through generate(): `is_prefill=True`, two voices of different length scattered into the prompts
    gv = torch.Generator().manual_seed(51)
    wavs = torch.zeros(2, 3200 * 3 + 100)
    wavs[0] = torch.randn(wavs.shape[1], generator=gv) * 0.05
    wavs[1, :3200 * 2 + 7] = torch.randn(3200 * 2 + 7, generator=gv) * 0.05
    vmasks = torch.zeros(2, 4, dtype=torch.bool)
    vmasks[0, :4] = True
    vmasks[1, :3] = True
    sim = torch.zeros(2, L0, dtype=torch.bool)
    sim[0, 3:7] = True                                             # 4 frames of voice 0 inside row 0
    sim[1, 6:9] = True                                             # 3 frames of voice 1 inside row 1 (after its 4 pad slots)
    ref_shim.script_tokens(L0, [_scripted(tok, "dddx"), _scripted(tok, "ddx")])
    torch.manual_seed(5)
    out = model.generate(input_ids=ids.clone(), attention_mask=mask.clone(), tokenizer=tok, cfg_scale=cfg_scale, max_new_tokens=40,
                         speech_tensors=wavs.clone(), speech_masks=vmasks.clone(), speech_input_mask=sim.clone(),
                         show_progress_bar=False, verbose=False, is_prefill=True)
    ref_shim.script_tokens()
    voice = dict(ids=ids, mask=mask, scripts=[_scripted(tok, "dddx"), _scripted(tok, "ddx")], max_new_tokens=40, seed=5,
                 max_length_times=2, refresh_negative=True, do_sample=False, wavs=wavs, voice_masks=vmasks, speech_input_mask=sim,
                 sequences=out.sequences.clone(), reach_max=out.reach_max_step_sample.clone(),
                 audio=[None if a is None else frame_sample(a) for a in out.speech_outputs])
    return dict(preset=preset, num_steps=steps, cfg_scale=cfg_scale, scripted=scripted, free=free, maxlen=maxlen, norefresh=norefresh,
                quirk=quirk, voice=voice, sampled=sampled, norefresh1=norefresh1, streamed=streamed, stopped=stopped, sde=sde)


def gen_streaming(ns, preset="tiny"):
    """The streaming-0.5B variant's own `generate()` (modeling_vibevoice_streaming_inference.py:412-725, loop body unmodified; same
    transformers-4.51.3 glue as `gen_loop`) on a synthetic split checkpoint: 1 lower + 1 upper layer of the tiny preset, random
    type embeddings and EOS classifier (`vv_streaming.streaming_state_dict`).  The four prefilled outputs the loop starts from are
    computed with the reference's own `forward_lm` / `forward_tts_lm` on a text-only prompt.  Cases:
      eos      classifier fires inside the first speech window (frames after it are dropped)
      windows  classifier biased off: three text windows (5,5,2), then text-less windows until max_new_tokens -> reach_max
      short    text shorter than one window, max length hit inside a speech window"""
    import importlib
    from oracle import vv_streaming as VS
    mod = ref_shim.install_streaming_generate_compat()
    scfg_mod = importlib.import_module("vibevoice.modular.configuration_vibevoice_streaming")
    cfg = preset_config(preset)
    rc = _ref_cfg(ns, cfg)
    tts_layers = 1
    sc = scfg_mod.VibeVoiceStreamingConfig(acoustic_tokenizer_config=rc.acoustic_tokenizer_config, decoder_config=rc.decoder_config,
                                            diffusion_head_config=rc.diffusion_head_config, tts_backbone_num_hidden_layers=tts_layers)
    sc.decoder_config._attn_implementation = "sdpa"
    tok = SynthTokenizer(cfg.decoder_config.vocab_size)
    tok.convert_tokens_to_ids = lambda t: tok.pad_token_id        # "<|image_pad|>" (:465)
    base = synth_state_dict(cfg, SEED, torch.float32)
    steps = 5
    out = dict(preset=preset, tts_layers=tts_layers, num_steps=steps, neg_id=tok.pad_token_id)
    g = torch.Generator().manual_seed(7)
    prompt = torch.randint(0, 2000, (1, 6), generator=g)
    for name, eos_bias, n_text, max_new, cfg_scale, seed in (("eos", -0.3, 12, 40, 1.5, 0), ("windows", -6.0, 12, 30, 1.5, 1),
                                                              ("short", -6.0, 3, 7, 1.3, 2)):
        sd = VS.streaming_state_dict(base, cfg, tts_layers, eos_bias=eos_bias)
        m = mod.VibeVoiceStreamingForConditionalGenerationInference(sc).eval()
        res = m.load_state_dict(sd, strict=False)
        assert not [k for k in res.missing_keys if "fix_std" not in k and "rotary" not in k] and not res.unexpected_keys, res
        m.set_ddpm_inference_steps(steps)
        text = torch.randint(0, 2000, (1, n_text), generator=g)
        neg = torch.full((1, 1), tok.pad_token_id)
        new = lambda: ref_shim.legacy_cache(sc.decoder_config)
        with torch.no_grad():
            lm = m.forward_lm(input_ids=prompt, attention_mask=torch.ones_like(prompt), past_key_values=new(), use_cache=True, return_dict=True)
            tts = m.forward_tts_lm(input_ids=prompt, attention_mask=torch.ones_like(prompt), past_key_values=new(), use_cache=True,
                                   return_dict=True, lm_last_hidden_state=lm.last_hidden_state, tts_text_masks=torch.ones_like(prompt))
            nlm = m.forward_lm(input_ids=neg, attention_mask=torch.ones_like(neg), past_key_values=new(), use_cache=True, return_dict=True)
            ntts = m.forward_tts_lm(input_ids=neg, attention_mask=torch.ones_like(neg), past_key_values=new(), use_cache=True,
                                    return_dict=True, lm_last_hidden_state=nlm.last_hidden_state, tts_text_masks=torch.ones_like(neg))
        # the caches grow inside generate(): keep what `all_prefilled_outputs` held at the call
        dump = lambda o: dict(kv=[(l.keys.clone(), l.values.clone()) for l in o.past_key_values.layers if l.keys is not None],
                              hidden=o.last_hidden_state.clone())
        pref = {k: dump(v) for k, v in (("lm", lm), ("tts_lm", tts), ("neg_lm", nlm), ("neg_tts_lm", ntts))}
        torch.manual_seed(seed)
        r = m.generate(input_ids=prompt.clone(), attention_mask=torch.ones_like(prompt), tts_lm_input_ids=prompt.clone(),
                       tts_lm_attention_mask=torch.ones_like(prompt), tts_text_ids=text.clone(),
                       all_prefilled_outputs={"lm": lm, "tts_lm": tts, "neg_lm": nlm, "neg_tts_lm": ntts}, tokenizer=tok,
                       cfg_scale=cfg_scale, max_new_tokens=max_new, show_progress_bar=False, verbose=False)
        out[name] = dict(prefilled=pref, eos_bias=eos_bias, prompt=prompt[0].clone(), text=text[0].clone(), max_new_tokens=max_new, cfg_scale=cfg_scale,
                         seed=seed, sequences=r.sequences.clone(), reach_max=r.reach_max_step_sample.clone(),
                         audio=None if r.speech_outputs[0] is None else r.speech_outputs[0].clone())
    return out


def gen_processor(ns):
    """The reference's `VibeVoiceProcessor` on the inputs of `tests/test_processor.py` (its stub tokenizer, script and voices):
    a batch of two scripts with voice prompts, and one script without."""
    import importlib
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_processor import SCRIPT, StubTokenizer, _voices
    rp = importlib.import_module("vibevoice.processor.vibevoice_processor")
    assert rp.__file__.startswith(ref_shim.REFERENCE_ROOT), rp.__file__
    ref = rp.VibeVoiceProcessor(tokenizer=StubTokenizer(), audio_processor=None)
    a = ref(text=[SCRIPT, "Speaker 0: Hi."], voice_samples=[_voices(), [_voices()[0]]], padding=True, return_tensors="pt")
    a2 = ref(text=SCRIPT, padding=True, return_tensors="pt")
    keys = ("input_ids", "attention_mask", "speech_input_mask", "speech_masks", "speech_tensors", "parsed_scripts")
    return dict(batch={k: a[k] for k in keys}, text_only={"input_ids": a2["input_ids"]})


GENERATORS = dict(processor=gen_processor, streaming=gen_streaming, loop=gen_loop, voice_prompt=gen_voice_prompt, scheduler=gen_scheduler, head=gen_head, codec=gen_codec, connector=gen_connector, lm=gen_lm)


def main():
    ns = ref_shim.load_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    only = set(sys.argv[1:])                  # `python -m oracle.make_golden loop` rewrites just that fixture
    for name, fn in GENERATORS.items():
        if only and name not in only:
            continue
        torch.manual_seed(0)
        data = fn(ns)
        path = os.path.join(GOLDEN_DIR, f"{name}.pt")
        torch.save(data, path)
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
