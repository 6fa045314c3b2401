"""`VibeVoiceProcessor` mirror: prompt layout, masks, left padding, voice-prompt token counts, wav round trip, and field-by-field
equality with the reference processor's output on the same inputs (`tests/golden/processor.pt`)."""
import os
import zlib

import numpy as np
import torch

from vibevoice_b200.processor import AudioNormalizer, VibeVoiceProcessor, load_wav_24k


class StubTokenizer:
    """Deterministic word-level tokenizer with the attributes the processors read (`modular_vibevoice_text_tokenizer.py:163-181`)."""
    speech_start_id, speech_end_id, speech_diffusion_id, pad_id, eos_token_id, bos_token_id = 9001, 9002, 9003, 9004, 9000, None
    pad_token_id = 9004

    def encode(self, text, add_special_tokens=True):
        out = []
        for piece in text.replace("\n", " \n ").split(" "):
            if piece:
                out.append(zlib.crc32(piece.encode()) % 8000)
        return out


SCRIPT = "Speaker 1: Hello there, how are you?\nSpeaker 2: Fine: thanks.\nSpeaker 1: Good."


def _voices():
    g = np.random.default_rng(0)
    return [g.standard_normal(3200 * 2 + 5).astype(np.float32) * 0.01, g.standard_normal(3200 * 3).astype(np.float32) * 0.3]


def test_prompt_layout_and_masks():
    p = VibeVoiceProcessor(tokenizer=StubTokenizer())
    out = p(text=[SCRIPT, "Speaker 0: Hi."], voice_samples=[_voices(), [_voices()[0]]], padding=True, return_tensors="pt")
    ids, att, sim = out["input_ids"], out["attention_mask"], out["speech_input_mask"]
    assert ids.shape == att.shape == sim.shape and ids.shape[0] == 2
    assert (ids[:, -1] == StubTokenizer.speech_start_id).all()                       # prompt ends with <speech_start>
    assert att[1, 0] == 0 and ids[1, 0] == StubTokenizer.pad_id and att[0].all()       # left padding with pad_id
    assert sim[0].sum() == 3 + 3 and sim[1].sum() == 3                                # ceil(len/3200) diffusion slots per voice
    assert (ids[0][sim[0]] == StubTokenizer.speech_diffusion_id).all()
    assert out["speech_tensors"].shape == (3, 9600) and out["speech_masks"].sum() == 9
    assert out["parsed_scripts"][0] == [(0, " Hello there, how are you?"), (1, " Fine: thanks."), (0, " Good.")]
    assert sorted(out["all_speakers_list"][0]) == [0, 1]
    rms = float(np.sqrt(np.mean(out["speech_tensors"][0, :6405].numpy() ** 2)))
    assert abs(20 * np.log10(rms) + 25) < 0.1                                          # -25 dBFS normalisation


def test_wav_io_roundtrip(tmp_path):
    from scipy.io import wavfile
    p = VibeVoiceProcessor(tokenizer=StubTokenizer())
    x = (np.sin(np.arange(16000) * 0.05) * 0.3).astype(np.float32)
    f16 = os.path.join(tmp_path, "v16k.wav")
    wavfile.write(f16, 16000, (x * 32767).astype(np.int16))
    y = load_wav_24k(f16)
    assert abs(len(y) - 24000) <= 1 and y.dtype == np.float32
    out = p.save_audio(torch.from_numpy(y)[None], output_path=os.path.join(tmp_path, "o", "out.wav"))
    sr, z = wavfile.read(out)
    assert sr == 24000 and len(z) == len(y)
    paths = p.save_audio([y, y[:100]], output_path=str(tmp_path))
    assert len(paths) == 2 and all(os.path.exists(q) for q in paths)


def test_matches_reference_processor(golden):
    """Field by field against what the reference processor returned for the same inputs (`oracle/make_golden.py::gen_processor`)."""
    g = golden("processor")
    mine = VibeVoiceProcessor(tokenizer=StubTokenizer())
    a = g["batch"]
    b = mine(text=[SCRIPT, "Speaker 0: Hi."], voice_samples=[_voices(), [_voices()[0]]], padding=True, return_tensors="pt")
    for k in ("input_ids", "attention_mask", "speech_input_mask", "speech_masks"):
        assert torch.equal(a[k], b[k]), k
    torch.testing.assert_close(a["speech_tensors"], b["speech_tensors"], rtol=1e-6, atol=1e-7)
    assert a["parsed_scripts"] == b["parsed_scripts"]
    b2 = mine(text=SCRIPT, padding=True, return_tensors="pt")
    assert torch.equal(g["text_only"]["input_ids"], b2["input_ids"]) and b2["speech_tensors"] is None


def test_convert_to_16_bit_wav_matches_the_gradio_helper():
    """`demo/gradio_demo.py:1058-1072`: int16 PCM, peak-normalised only when the signal leaves [-1, 1]."""
    from vibevoice_b200.processor import convert_to_16_bit_wav
    x = torch.tensor([[0.0, 0.5, -1.0, 0.25]])
    assert convert_to_16_bit_wav(x).tolist() == [[0, 16383, -32767, 8191]]
    y = np.array([0.0, 2.0, -4.0])
    assert convert_to_16_bit_wav(y).tolist() == [0, 16383, -32767]
    assert convert_to_16_bit_wav(x).dtype == np.int16
