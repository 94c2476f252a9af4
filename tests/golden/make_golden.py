"""Generate the golden vectors in this directory by running the UNMODIFIED reference
(/root/reference, yeyupiaoling/MASR @ fe0010de) in the build container through
``oracle/ref_shims.py``.  The reference has no tests or golden vectors of its own (SURVEY.md §4),
and it cannot travel to the GPU box, so its outputs on deterministic synthetic inputs are frozen here.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz / *.json

Inputs are regenerated from seeds by ``masr_b200.synth`` (weights, vocabulary, CMVN, audio), so only
the reference's OUTPUTS are stored.
"""
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
HERE = os.path.dirname(os.path.abspath(__file__))

from oracle import ref_shims  # noqa: E402

ref_shims.install()

import torch  # noqa: E402
import yaml  # noqa: E402

from masr_b200 import synth  # noqa: E402

V = synth.DEFAULT_VOCAB_SIZE

# (name, kind, seed, num_samples[, scale])
FBANK_CASES = [
    ("noise_1s", "noise", 0, 16000),
    ("speech_0p7s", "speech", 1, 11200),
    ("speech_min", "speech", 2, 400),          # exactly one frame
    ("speech_loud", "speech", 3, 8000, 30.0),  # clips at int16 after normalisation? (exercises the clamp path)
    ("speech_quiet", "speech", 4, 8000, 1e-3),
]

ENCODER_CASES = [  # (name, streaming, weight seed, audio kind, audio seed, samples)
    ("causal_speech_1p5s", True, 0, "speech", 10, 24000),
    ("causal_noise_1s", True, 0, "noise", 11, 16000),
    ("noncausal_speech_1p2s", False, 1, "speech", 12, 19200),
]

EFFICIENT_CASES = [  # (name, streaming, weight seed, audio kind, audio seed, samples)
    ("eff_causal_speech_2s", True, 0, "speech", 20, 32000),
    ("eff_noncausal_speech_1p3s", False, 1, "speech", 21, 20800 + 37),
]

SQUEEZE_CASES = [  # (name, streaming, weight seed, audio kind, audio seed, samples)
    ("sqz_causal_speech_2s", True, 0, "speech", 25, 32000),
    ("sqz_noncausal_speech_1p3s", False, 1, "speech", 26, 20800 + 37),
]

DS2_CASES = [  # (name, streaming, weight seed, audio kind, audio seed, samples)
    ("ds2_uni_speech_1p5s", True, 0, "speech", 35, 24000),
    ("ds2_bi_speech_1p2s", False, 1, "speech", 36, 19200 + 80),
]

STREAM_CASE = ("stream_speech_3p4s", 0, "speech", 30, 54400, 8000)  # weight seed, kind, audio seed, samples, push


def make_audio(kind, seed, n, scale=1.0):
    x = synth.noise_audio(seed, n) if kind == "noise" else synth.speechlike_audio(seed, n)
    return (x * np.float32(scale)).astype(np.float32)


def build_reference_model(tmp, streaming, wseed):
    from masr.model_utils.conformer.model import ConformerModel
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "conformer.yml"), encoding="utf-8"))
    mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
    synth.write_mean_istd(mi, wseed)
    model = ConformerModel(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=streaming,
                           encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"], **cfg["model_conf"])
    sd = synth.to_torch(synth.conformer_state_dict(wseed, V))
    res = model.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys and all(k.startswith("decoder.") for k in res.missing_keys)
    return model.eval(), cfg, mi


def gen_fbank():
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    out = {}
    meta = []
    for case in FBANK_CASES:
        name, kind, seed, n = case[:4]
        scale = case[4] if len(case) > 4 else 1.0
        x = make_audio(kind, seed, n, scale)
        seg = AudioSegment.from_ndarray(x.copy(), 16000)
        feat = af.featurize(seg)                 # normalises seg in place
        q = seg.to("int16")
        out[name + "/feat"] = np.asarray(feat, np.float32)
        out[name + "/int16"] = q
        meta.append({"name": name, "kind": kind, "seed": seed, "samples": n, "scale": scale})
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
    np.savez_compressed(os.path.join(HERE, "fbank_golden.npz"), **out)
    print("fbank_golden.npz", {k: v.shape for k, v in out.items() if k != "meta"})


def gen_encoder(tmp):
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    from masr.decoders.ctc_greedy_decoder import greedy_decoder
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    vocab = synth.vocabulary(V)
    out, meta = {}, []
    for name, streaming, wseed, kind, aseed, n in ENCODER_CASES:
        model, _, _ = build_reference_model(tmp, streaming, wseed)
        scripted = model.export()                # TorchScript, as MASRTrainer.export does (trainer.py:684)
        x = make_audio(kind, aseed, n)
        feat = torch.from_numpy(af.featurize(AudioSegment.from_ndarray(x.copy(), 16000)))[None]
        with torch.no_grad():
            probs = scripted.get_encoder_out(feat, torch.tensor([feat.shape[1]]))[0]
            enc, _ = model.encoder(feat, torch.tensor([feat.shape[1]]), decoding_chunk_size=-1, num_decoding_left_chunks=-1)
        score, text = greedy_decoder(probs.numpy(), vocab)
        top = probs.topk(8, dim=1)
        out[name + "/feat"] = feat[0].numpy()
        out[name + "/enc"] = enc[0].numpy()
        out[name + "/top_p"] = top.values.numpy()
        out[name + "/top_i"] = top.indices.numpy().astype(np.int32)
        out[name + "/ids"] = probs.argmax(1).numpy().astype(np.int32)
        meta.append({"name": name, "streaming": streaming, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n,
                     "score": score, "text": text})
        print(name, "T", probs.shape[0], "score", score, "text", text)
    out["meta"] = np.frombuffer(json.dumps(meta, ensure_ascii=False).encode("utf-8"), np.uint8)
    np.savez_compressed(os.path.join(HERE, "conformer_golden.npz"), **out)


def gen_efficient(tmp):
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    from masr.decoders.ctc_greedy_decoder import greedy_decoder
    from masr.model_utils.efficient_conformer.model import EfficientConformerModel
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "efficient_conformer.yml"), encoding="utf-8"))
    vocab = synth.vocabulary(V)
    out, meta = {}, []
    for name, streaming, wseed, kind, aseed, n in EFFICIENT_CASES:
        mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
        synth.write_mean_istd(mi, wseed)
        model = EfficientConformerModel(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=streaming,
                                        encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"], **cfg["model_conf"])
        res = model.load_state_dict(synth.to_torch(synth.efficient_conformer_state_dict(wseed, V)), strict=False)
        assert not res.unexpected_keys and all(k.startswith("decoder.") for k in res.missing_keys)
        scripted = model.eval().export()
        x = make_audio(kind, aseed, n)
        feat = torch.from_numpy(af.featurize(AudioSegment.from_ndarray(x.copy(), 16000)))[None]
        with torch.no_grad():
            probs = scripted.get_encoder_out(feat, torch.tensor([feat.shape[1]]))[0]
        score, text = greedy_decoder(probs.numpy(), vocab)
        top = probs.topk(8, dim=1)
        out[name + "/feat"] = feat[0].numpy()
        out[name + "/top_p"] = top.values.numpy()
        out[name + "/top_i"] = top.indices.numpy().astype(np.int32)
        out[name + "/ids"] = probs.argmax(1).numpy().astype(np.int32)
        meta.append({"name": name, "streaming": streaming, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n,
                     "score": score, "text": text})
        print(name, "T", probs.shape[0], "score", score, "text", text)
    out["meta"] = np.frombuffer(json.dumps(meta, ensure_ascii=False).encode("utf-8"), np.uint8)
    np.savez_compressed(os.path.join(HERE, "efficient_golden.npz"), **out)


def gen_squeezeformer(tmp):
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    from masr.decoders.ctc_greedy_decoder import greedy_decoder
    from masr.model_utils.squeezeformer.model import SqueezeformerModel
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "squeezeformer.yml"), encoding="utf-8"))
    vocab = synth.vocabulary(V)
    out, meta = {}, []
    for name, streaming, wseed, kind, aseed, n in SQUEEZE_CASES:
        mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
        synth.write_mean_istd(mi, wseed)
        model = SqueezeformerModel(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=streaming,
                                   encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"], **cfg["model_conf"])
        res = model.load_state_dict(synth.to_torch(synth.squeezeformer_state_dict(wseed, V, streaming=streaming)), strict=False)
        assert not res.unexpected_keys and all(k.startswith("decoder.") for k in res.missing_keys)
        scripted = model.eval().export()
        x = make_audio(kind, aseed, n)
        feat = torch.from_numpy(af.featurize(AudioSegment.from_ndarray(x.copy(), 16000)))[None]
        with torch.no_grad():
            probs = scripted.get_encoder_out(feat, torch.tensor([feat.shape[1]]))[0]
        score, text = greedy_decoder(probs.numpy(), vocab)
        top = probs.topk(8, dim=1)
        out[name + "/feat"] = feat[0].numpy()
        out[name + "/top_p"] = top.values.numpy()
        out[name + "/top_i"] = top.indices.numpy().astype(np.int32)
        out[name + "/ids"] = probs.argmax(1).numpy().astype(np.int32)
        meta.append({"name": name, "streaming": streaming, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n,
                     "score": score, "text": text})
        print(name, "T", probs.shape[0], "score", score, "text", text)
    out["meta"] = np.frombuffer(json.dumps(meta, ensure_ascii=False).encode("utf-8"), np.uint8)
    np.savez_compressed(os.path.join(HERE, "squeezeformer_golden.npz"), **out)


def gen_deepspeech2(tmp):
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    from masr.decoders.ctc_greedy_decoder import greedy_decoder
    from masr.model_utils.deepspeech2.model import DeepSpeech2Model
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "deepspeech2.yml"), encoding="utf-8"))
    vocab = synth.vocabulary(V)
    out, meta = {}, []
    for name, streaming, wseed, kind, aseed, n in DS2_CASES:
        mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
        synth.write_mean_istd(mi, wseed)
        model = DeepSpeech2Model(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=streaming,
                                 encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"])
        res = model.load_state_dict(synth.to_torch(synth.deepspeech2_state_dict(wseed, V, streaming=streaming)), strict=True)
        scripted = model.eval().export()
        x = make_audio(kind, aseed, n)
        feat = torch.from_numpy(af.featurize(AudioSegment.from_ndarray(x.copy(), 16000)))[None]
        with torch.no_grad():
            probs = scripted.get_encoder_out(feat, torch.tensor([feat.shape[1]]))[0]
        score, text = greedy_decoder(probs.numpy(), vocab)
        top = probs.topk(8, dim=1)
        out[name + "/feat"] = feat[0].numpy()
        out[name + "/top_p"] = top.values.numpy()
        out[name + "/top_i"] = top.indices.numpy().astype(np.int32)
        out[name + "/ids"] = probs.argmax(1).numpy().astype(np.int32)
        meta.append({"name": name, "streaming": streaming, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n,
                     "score": score, "text": text})
        print(name, "T", probs.shape[0], "score", score, "text", text)
    out["meta"] = np.frombuffer(json.dumps(meta, ensure_ascii=False).encode("utf-8"), np.uint8)
    np.savez_compressed(os.path.join(HERE, "deepspeech2_golden.npz"), **out)


def gen_predictor(tmp):
    """The real ``MASRPredictor`` end to end (greedy): whole-utterance and streaming pushes."""
    from masr.predict import MASRPredictor
    name, wseed, kind, aseed, n, push = STREAM_CASE
    model, cfg, mi = build_reference_model(tmp, True, wseed)
    mp = os.path.join(tmp, "inference.pt")
    torch.jit.save(model.export(), mp)
    vp = os.path.join(tmp, "vocabulary.txt")
    synth.write_vocabulary(vp, V)
    cfg["dataset_conf"]["dataset_vocab"] = vp
    cfg["dataset_conf"]["mean_istd_path"] = mi
    cfg["decoder"] = "ctc_greedy"
    np.random.seed(0)
    pred = MASRPredictor(configs=cfg, model_path=mp, use_gpu=False)
    x = make_audio(kind, aseed, n)
    whole = pred.predict(audio_data=x.copy())
    pcm = (np.clip(x, -1, 1) * 32767).astype("<i2")
    pushes = []
    pred.reset_stream()
    for s in range(0, len(pcm), push):
        chunk = pcm[s:s + push].tobytes()
        is_end = s + push >= len(pcm)
        r = pred.predict_stream(audio_data=chunk, is_end=is_end)
        pushes.append(None if r is None else {"text": r["text"], "score": r["score"]})
    pred.reset_stream()
    # second run with float ndarray pushes, to pin reset_stream + the ndarray path
    pushes_nd = []
    for s in range(0, len(x), push):
        r = pred.predict_stream(audio_data=x[s:s + push].copy(), is_end=s + push >= len(x))
        pushes_nd.append(None if r is None else {"text": r["text"], "score": r["score"]})
    data = {"name": name, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n, "push": push,
            "whole": whole, "pushes_pcm": pushes, "pushes_ndarray": pushes_nd}
    with open(os.path.join(HERE, "predictor_golden.json"), "w", encoding="utf-8") as f:
        json.dump(data, f, ensure_ascii=False, indent=1)
    print("predictor whole", whole)
    print("pushes", pushes)


def build_reference_squeezeformer(tmp, streaming, wseed):
    from masr.model_utils.squeezeformer.model import SqueezeformerModel
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "squeezeformer.yml"), encoding="utf-8"))
    mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
    synth.write_mean_istd(mi, wseed)
    model = SqueezeformerModel(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=streaming,
                               encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"], **cfg["model_conf"])
    res = model.load_state_dict(synth.to_torch(synth.squeezeformer_state_dict(wseed, V, streaming=streaming)), strict=False)
    assert not res.unexpected_keys and all(k.startswith("decoder.") for k in res.missing_keys)
    return model.eval(), cfg, mi


SQZ_STREAM_CASE = ("sqz_stream_speech_3p7s", 0, "speech", 31, 59200 + 123, 8000)  # weight seed, kind, audio seed, samples, push


def gen_predictor_squeezeformer(tmp):
    """The real ``MASRPredictor`` with the streaming Squeezeformer (greedy): whole utterance, PCM pushes (the last chunk is
    short) and per-chunk frame ids of ``get_encoder_out_chunk``."""
    from masr.predict import MASRPredictor
    name, wseed, kind, aseed, n, push = SQZ_STREAM_CASE
    model, cfg, mi = build_reference_squeezeformer(tmp, True, wseed)
    mp = os.path.join(tmp, "inference_sqz.pt")
    torch.jit.save(model.export(), mp)
    vp = os.path.join(tmp, "vocabulary.txt")
    synth.write_vocabulary(vp, V)
    cfg["dataset_conf"]["dataset_vocab"] = vp
    cfg["dataset_conf"]["mean_istd_path"] = mi
    cfg["decoder"] = "ctc_greedy"
    np.random.seed(0)
    pred = MASRPredictor(configs=cfg, model_path=mp, use_gpu=False)
    x = make_audio(kind, aseed, n)
    whole = pred.predict(audio_data=x.copy())
    pcm = (np.clip(x, -1, 1) * 32767).astype("<i2")
    pushes = []
    pred.reset_stream()
    for s in range(0, len(pcm), push):
        r = pred.predict_stream(audio_data=pcm[s:s + push].tobytes(), is_end=s + push >= len(pcm))
        pushes.append(None if r is None else {"text": r["text"], "score": r["score"]})
    pred.reset_stream()
    data = {"name": name, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n, "push": push,
            "whole": whole, "pushes_pcm": pushes}
    with open(os.path.join(HERE, "predictor_golden_squeezeformer.json"), "w", encoding="utf-8") as f:
        json.dump(data, f, ensure_ascii=False, indent=1)
    print("squeezeformer predictor whole", whole)
    print("pushes", pushes)


EFF_STREAM_CASE = ("eff_stream_speech_3p6s", 0, "speech", 32, 57600 + 77, 8000)  # weight seed, kind, audio seed, samples, push


def gen_predictor_efficient(tmp):
    """The real ``MASRPredictor`` with the streaming EfficientConformer (greedy): whole utterance and PCM pushes."""
    from masr.model_utils.efficient_conformer.model import EfficientConformerModel
    from masr.predict import MASRPredictor
    name, wseed, kind, aseed, n, push = EFF_STREAM_CASE
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "efficient_conformer.yml"), encoding="utf-8"))
    mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
    synth.write_mean_istd(mi, wseed)
    model = EfficientConformerModel(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=True,
                                    encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"], **cfg["model_conf"])
    res = model.load_state_dict(synth.to_torch(synth.efficient_conformer_state_dict(wseed, V)), strict=False)
    assert not res.unexpected_keys and all(k.startswith("decoder.") for k in res.missing_keys)
    mp = os.path.join(tmp, "inference_eff.pt")
    torch.jit.save(model.eval().export(), mp)
    vp = os.path.join(tmp, "vocabulary.txt")
    synth.write_vocabulary(vp, V)
    cfg["dataset_conf"]["dataset_vocab"] = vp
    cfg["dataset_conf"]["mean_istd_path"] = mi
    cfg["decoder"] = "ctc_greedy"
    cfg["streaming"] = True
    np.random.seed(0)
    pred = MASRPredictor(configs=cfg, model_path=mp, use_gpu=False)
    x = make_audio(kind, aseed, n)
    whole = pred.predict(audio_data=x.copy())
    pcm = (np.clip(x, -1, 1) * 32767).astype("<i2")
    pushes = []
    pred.reset_stream()
    for s in range(0, len(pcm), push):
        r = pred.predict_stream(audio_data=pcm[s:s + push].tobytes(), is_end=s + push >= len(pcm))
        pushes.append(None if r is None else {"text": r["text"], "score": r["score"]})
    pred.reset_stream()
    data = {"name": name, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n, "push": push,
            "whole": whole, "pushes_pcm": pushes}
    with open(os.path.join(HERE, "predictor_golden_efficient.json"), "w", encoding="utf-8") as f:
        json.dump(data, f, ensure_ascii=False, indent=1)
    print("efficient predictor whole", whole)
    print("pushes", pushes)


DS2_STREAM_CASE = ("ds2_stream_speech_3p75s", 0, "speech", 33, 60000, 8000)  # weight seed, kind, audio seed, samples, push


def gen_predictor_deepspeech2(tmp):
    """The real ``MASRPredictor`` with the streaming (unidirectional) DeepSpeech2, greedy: whole utterance and PCM pushes."""
    from masr.model_utils.deepspeech2.model import DeepSpeech2Model
    from masr.predict import MASRPredictor
    name, wseed, kind, aseed, n, push = DS2_STREAM_CASE
    cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", "deepspeech2.yml"), encoding="utf-8"))
    mi = os.path.join(tmp, f"mean_istd_{wseed}.json")
    synth.write_mean_istd(mi, wseed)
    model = DeepSpeech2Model(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=True,
                             encoder_conf=cfg["encoder_conf"], decoder_conf=cfg["decoder_conf"])
    model.load_state_dict(synth.to_torch(synth.deepspeech2_state_dict(wseed, V, streaming=True)), strict=True)
    mp = os.path.join(tmp, "inference_ds2.pt")
    torch.jit.save(model.eval().export(), mp)
    vp = os.path.join(tmp, "vocabulary.txt")
    synth.write_vocabulary(vp, V)
    cfg["dataset_conf"]["dataset_vocab"] = vp
    cfg["dataset_conf"]["mean_istd_path"] = mi
    cfg["decoder"] = "ctc_greedy"
    cfg["streaming"] = True
    np.random.seed(0)
    pred = MASRPredictor(configs=cfg, model_path=mp, use_gpu=False)
    x = make_audio(kind, aseed, n)
    whole = pred.predict(audio_data=x.copy())
    pcm = (np.clip(x, -1, 1) * 32767).astype("<i2")
    pushes = []
    pred.reset_stream()
    for s in range(0, len(pcm), push):
        r = pred.predict_stream(audio_data=pcm[s:s + push].tobytes(), is_end=s + push >= len(pcm))
        pushes.append(None if r is None else {"text": r["text"], "score": r["score"]})
    pred.reset_stream()
    data = {"name": name, "wseed": wseed, "kind": kind, "aseed": aseed, "samples": n, "push": push,
            "whole": whole, "pushes_pcm": pushes}
    with open(os.path.join(HERE, "predictor_golden_deepspeech2.json"), "w", encoding="utf-8") as f:
        json.dump(data, f, ensure_ascii=False, indent=1)
    print("deepspeech2 predictor whole", whole)
    print("pushes", pushes)


def vad_prob_cases():
    """Deterministic per-window speech-probability tracks (what the silero network would emit) exercising every branch of
    the segmentation state machine: short blips (< min speech), short dips (< min silence), adjacent segments closer than
    two pads, speech running to the end of the audio, an empty track."""
    rng = np.random.default_rng(7)
    cases = []
    for k in range(6):
        n = int(rng.integers(40, 400))
        p = np.clip(rng.normal(0.2, 0.1, n), 0, 1)
        pos = 0
        while pos < n:
            gap, run = int(rng.integers(1, 40)), int(rng.integers(1, 60))
            pos += gap
            p[pos:pos + run] = np.clip(rng.normal(0.85, 0.1, max(0, min(n, pos + run) - pos)), 0, 1)
            pos += run
        if k == 1:
            p[-30:] = 0.9                                  # speech until the end
        if k == 2:
            p[:] = 0.1                                     # no speech at all
        tail = int(rng.integers(0, 512))
        cases.append({"probs": [float(np.float32(v)) for v in p], "samples": (n - 1) * 512 + (tail or 512)})
    return cases


def gen_vad():
    """``VADPredictor.get_speech_timestamps`` (vad_predictor.py:106-175) with the ONNX network replaced by a scripted
    probability track: freezes the segmentation state machine of predict_long (SURVEY §8 f4)."""
    import types
    sys.modules.setdefault("onnxruntime", types.ModuleType("onnxruntime"))
    from masr.infer_utils.vad_predictor import VADPredictor
    out = []
    for case in vad_prob_cases():
        for kw in ({}, {"threshold": 0.6, "min_speech_duration_ms": 100, "min_silence_duration_ms": 300, "speech_pad_ms": 100}):
            v = object.__new__(VADPredictor)
            v.threshold, v.min_speech_duration_ms = kw.get("threshold", 0.5), kw.get("min_speech_duration_ms", 250)
            v.min_silence_duration_ms, v.window_size_samples = kw.get("min_silence_duration_ms", 100), 512
            v.speech_pad_ms = kw.get("speech_pad_ms", 30)
            it = iter(case["probs"])
            VADPredictor.reset_states(v)
            v.__class__ = type("ScriptedVAD", (VADPredictor,), {"__call__": lambda self, x, sr, it=it: np.float32(next(it))})
            ts = v.get_speech_timestamps(np.zeros(case["samples"], np.float32), 16000)
            out.append({"probs": case["probs"], "samples": case["samples"], "kw": kw, "timestamps": ts})
    with open(os.path.join(HERE, "vad_timestamps_golden.json"), "w", encoding="utf-8") as f:
        json.dump(out, f)
    print("vad cases", [(len(c["probs"]), len(c["timestamps"])) for c in out])


def sample_array(out, key, a, n=128, top_k=0):
    """Store a fixed sample of ``a``: its shape, ``n`` flat positions drawn with a fixed seed and (``top_k`` > 0, for
    probabilities [..., V]) every row's argmax and ``top_k`` largest entries, where fp32 differences are largest.
    Keeps a chunk's [T, 4233] posteriors and its caches to a few KB each."""
    a = np.ascontiguousarray(np.asarray(a, np.float32))
    flat = a.reshape(-1)
    idx = np.arange(flat.size) if flat.size <= n else np.random.default_rng(len(out)).choice(flat.size, n, replace=False)
    if top_k:
        rows = a.reshape(-1, a.shape[-1])
        top = np.argsort(-rows, axis=1, kind="stable")[:, :top_k]
        idx = np.concatenate([idx, (np.arange(rows.shape[0])[:, None] * rows.shape[1] + top).reshape(-1)])
        out[key + "/ids"] = rows.argmax(1).astype(np.int32)
    idx = np.unique(idx)
    out[key + "/shape"] = np.asarray(a.shape, np.int64)
    out[key + "/idx"] = idx.astype(np.int32)
    out[key + "/val"] = flat[idx]


def gen_reference_chunks(tmp):
    """The reference's featurizer, the Conformer's whole-utterance forward and the chunk-by-chunk forward of every
    streaming model (posteriors and both caches after each chunk, the last chunk short), sampled by ``sample_array``.
    Frozen so that tests/test_oracle_vs_reference.py can check the oracle's chunk paths without the reference."""
    from masr.data_utils.audio import AudioSegment
    from masr.data_utils.featurizer.audio_featurizer import AudioFeaturizer
    from masr.model_utils.deepspeech2.model import DeepSpeech2Model
    from masr.model_utils.efficient_conformer.model import EfficientConformerModel
    from masr.model_utils.squeezeformer.model import SqueezeformerModel
    from oracle import fbank as ob
    out = {}
    af = AudioFeaturizer(feature_method="fbank", n_mels=80, sample_rate=16000, use_dB_normalization=True, target_dB=-20)
    for kind, seed, n in [("noise", 5, 20000), ("speech", 6, 33333)]:
        feat = af.featurize(AudioSegment.from_ndarray(make_audio(kind, seed, n), 16000))
        sample_array(out, f"fbank/{kind}_{seed}", feat, n=1024)
    pcm = (make_audio("speech", 7, 8000) * 20000).astype(np.int16)
    sample_array(out, "fbank/pcm_speech_7", af.featurize(AudioSegment.from_pcm_bytes(pcm.tobytes())), n=1024)

    def featurize(kind, seed, n):
        return torch.from_numpy(ob.featurize(make_audio(kind, seed, n)))[None]

    def build(cls, yml, sdn, strict=False, model_conf=True):
        cfg = yaml.safe_load(open(os.path.join(ref_shims.REFERENCE_ROOT, "configs", yml), encoding="utf-8"))
        mi = os.path.join(tmp, "mi.json")
        synth.write_mean_istd(mi, 0)
        m = cls(input_dim=80, vocab_size=V, mean_istd_path=mi, streaming=True, encoder_conf=cfg["encoder_conf"],
                decoder_conf=cfg["decoder_conf"], **(cfg["model_conf"] if model_conf else {})).eval()
        m.load_state_dict(synth.to_torch(sdn), strict=strict)
        return m

    def attention_chunks(name, m, feat, first_len):
        att = torch.zeros(0, 0, 0, 0)
        cnn = torch.zeros(0, 0, 0, 0)
        off = 0
        nf = feat.shape[1]
        for i, cur in enumerate(range(0, nf - first_len + 1, 64)):
            pr, att, cnn = m.get_encoder_out_chunk(feat[:, cur:min(cur + 67, nf)], off, -16, att, cnn)
            off += pr.shape[1]
            sample_array(out, f"{name}/{i}/probs", pr, top_k=4)
            sample_array(out, f"{name}/{i}/att", att)
            sample_array(out, f"{name}/{i}/cnn", cnn)

    with torch.no_grad():
        m, _, _ = build_reference_model(tmp, True, 0)
        feat = featurize("speech", 8, 16000 * 3)
        sample_array(out, "conformer/full", m.get_encoder_out(feat, torch.tensor([feat.shape[1]])), n=1024, top_k=8)
        attention_chunks("conformer", m, feat, 67)
        m = build(SqueezeformerModel, "squeezeformer.yml", synth.squeezeformer_state_dict(0, V, streaming=True))
        attention_chunks("squeezeformer", m, featurize("speech", 9, 16000 * 3 + 4000), 7)
        m = build(EfficientConformerModel, "efficient_conformer.yml", synth.efficient_conformer_state_dict(0, V))
        attention_chunks("efficient", m, featurize("speech", 13, 16000 * 3 + 4000), 7)
        m = build(DeepSpeech2Model, "deepspeech2.yml", synth.deepspeech2_state_dict(0, V, streaming=True), strict=True,
                  model_conf=False)
        feat = featurize("speech", 14, 16000 * 3 + 4000)
        h = torch.zeros(0, 0, 0, 0)
        c = torch.zeros(0, 0, 0, 0)
        nf = feat.shape[1]
        for i, cur in enumerate(range(0, nf - 7 + 1, 64)):
            ch = feat[:, cur:min(cur + 67, nf)]
            pr, lens, h, c = m.get_encoder_out_chunk(ch, torch.tensor([ch.shape[1]]), h, c)
            out[f"deepspeech2/{i}/len"] = lens.numpy().astype(np.int64)
            sample_array(out, f"deepspeech2/{i}/probs", pr[0], top_k=4)
            sample_array(out, f"deepspeech2/{i}/h", h.reshape(-1))
            sample_array(out, f"deepspeech2/{i}/c", c.reshape(-1))
    np.savez_compressed(os.path.join(HERE, "reference_chunks_golden.npz"), **out)
    print("reference_chunks_golden.npz", len(out), "arrays")


if __name__ == "__main__":
    torch.set_num_threads(8)
    with tempfile.TemporaryDirectory() as tmp:
        which = sys.argv[1:] or ["fbank", "encoder", "predictor", "efficient", "squeezeformer", "deepspeech2",
                                  "predictor_squeezeformer", "predictor_efficient", "predictor_deepspeech2", "vad",
                                  "reference_chunks"]
        if "reference_chunks" in which:
            gen_reference_chunks(tmp)
        if "deepspeech2" in which:
            gen_deepspeech2(tmp)
        if "squeezeformer" in which:
            gen_squeezeformer(tmp)
        if "fbank" in which:
            gen_fbank()
        if "encoder" in which:
            gen_encoder(tmp)
        if "predictor" in which:
            gen_predictor(tmp)
        if "predictor_squeezeformer" in which:
            gen_predictor_squeezeformer(tmp)
        if "predictor_efficient" in which:
            gen_predictor_efficient(tmp)
        if "predictor_deepspeech2" in which:
            gen_predictor_deepspeech2(tmp)
        if "efficient" in which:
            gen_efficient(tmp)
        if "vad" in which:
            gen_vad()
