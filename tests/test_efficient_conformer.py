"""EfficientConformer: oracle pinned to the reference's frozen outputs (CPU) and the CUDA engine against
oracle + golden (GPU)."""
import numpy as np
import pytest
import torch

from conftest import load_npz, make_audio
from masr_b200 import synth
from oracle import conformer as oc, ctc as octc, efficient_conformer as oe, fbank as ob

_W = {}


def weights(seed):
    if seed not in _W:
        _W[seed] = synth.efficient_conformer_state_dict(seed)
    return _W[seed]


def test_oracle_matches_reference_golden():
    z, meta = load_npz("efficient_golden.npz")
    vocab = synth.vocabulary()
    for m in meta:
        sd = synth.to_torch(weights(m["wseed"]))
        cfg = oe.EfficientConfig(causal=m["streaming"])
        feat = torch.from_numpy(z[m["name"] + "/feat"])[None]
        with torch.no_grad():
            probs = oe.get_encoder_out(sd, cfg, feat)[0].numpy()
        assert probs.shape[0] == z[m["name"] + "/ids"].shape[0]          # 80 ms frames: ceil(T/2)
        assert np.array_equal(probs.argmax(1), z[m["name"] + "/ids"])
        got = np.take_along_axis(probs, z[m["name"] + "/top_i"].astype(np.int64), axis=1)
        assert np.abs(got - z[m["name"] + "/top_p"]).max() < 5e-6     # fp32 sums run in another order on another CPU
        score, text, _ = octc.greedy_decode(probs, vocab)
        assert text == m["text"] and abs(score - m["score"]) < 1e-4


def test_grouping_is_a_memory_view():
    """pad4group's regrouping == reading 3 consecutive 256-float frames as 4 heads x 192 (what the kernel does)."""
    T, d, h, g = 8, 256, 4, 3
    q = torch.arange(T * d, dtype=torch.float32).view(1, T, d)
    pad = (g - T % g) % g
    ref = torch.nn.functional.pad(q.view(1, T, h, d // h).transpose(1, 2), (0, 0, 0, pad))      # [1,h,T+pad,dk] like the reference
    ref = ref.transpose(1, 2).contiguous().view(1, -1, h, (d // h) * g).transpose(1, 2)          # attention.py:58
    flat = torch.nn.functional.pad(q, (0, 0, 0, pad)).view(-1)
    for j in range(ref.shape[2]):
        for hh in range(h):
            assert torch.equal(ref[0, hh, j], flat[j * g * d + hh * 192: j * g * d + (hh + 1) * 192])


@pytest.mark.gpu
@pytest.mark.parametrize("streaming,wseed", [(True, 0), (False, 1)])
def test_gpu_engine_matches_oracle_and_golden(streaming, wseed):
    from masr_b200.engine import EfficientConformerEngine
    eng = EfficientConformerEngine(weights(wseed), streaming=streaming)
    sd = synth.to_torch(weights(wseed))
    cfg = oe.EfficientConfig(causal=streaming)
    vocab = synth.vocabulary()
    z, meta = load_npz("efficient_golden.npz")
    for m in meta:
        if m["streaming"] != streaming:
            continue
        feat = z[m["name"] + "/feat"]
        res = eng.transcribe_features(torch.from_numpy(feat)[None].to(eng.device), [feat.shape[0]], None, return_frames=True)
        assert np.array_equal(res.frame_ids[0, :res.frame_lens[0]], z[m["name"] + "/ids"])
        assert "".join(vocab[i] for i in res.tokens[0]).replace("<space>", " ") == m["text"]
        assert abs(res.scores[0] - m["score"]) < 1e-3
        probs = eng.posteriors(feat[None], [feat.shape[0]])[0]
        got = np.take_along_axis(probs, z[m["name"] + "/top_i"].astype(np.int64), axis=1)
        assert np.abs(got - z[m["name"] + "/top_p"]).max() < 2e-5
    # ragged batch, B=1 semantics per row (lengths chosen to hit T % 3 in {0,1,2} and odd/even T)
    lens = [16000 * 3 + 17, 9000, 16000 * 2, 400 + 160 * 30, 16000 * 4 + 800, 16000 + 320]
    waves = [make_audio("speech" if i % 2 == 0 else "noise", 70 + i, n) for i, n in enumerate(lens)]
    res = eng.transcribe(waves, return_frames=True)
    for i, w in enumerate(waves):
        f = torch.from_numpy(ob.featurize(w.copy()))
        with torch.no_grad():
            probs = oe.get_encoder_out(sd, cfg, f[None])[0].numpy()
        n = res.frame_lens[i]
        assert n == probs.shape[0]
        assert np.array_equal(probs.argmax(1), res.frame_ids[i, :n]), i
        score, text, toks = octc.greedy_decode(probs, vocab)
        assert toks == res.tokens[i] and abs(score - res.scores[i]) < 1e-3
