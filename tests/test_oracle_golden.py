"""CPU: the oracle restatement is pinned to the reference's frozen outputs (tests/golden/*, made by
tests/golden/make_golden.py from the unmodified reference)."""
import numpy as np
import torch

from conftest import make_audio, synth_weights
from masr_b200 import synth
from oracle import conformer as oc, ctc as octc, fbank as ob

FBANK_TOL = 5e-4      # log-mel domain; the FFT (pocketfft float32 here vs torch's) is the noise floor ~1e-4


def test_fbank_oracle_matches_reference(fbank_golden):
    z, meta = fbank_golden
    for m in meta:
        x = make_audio(m["kind"], m["seed"], m["samples"], m["scale"])
        xf = ob.to_float32(x)
        y, _ = ob.normalize_gain(xf)
        q = ob.to_int16(y)
        assert np.array_equal(q, z[m["name"] + "/int16"]), m["name"]     # integer work: bit-exact
        feat = ob.kaldi_fbank(q)
        ref = z[m["name"] + "/feat"]
        assert feat.shape == ref.shape
        assert np.abs(feat - ref).max() < FBANK_TOL, (m["name"], np.abs(feat - ref).max())


def test_fbank_frame_count_and_short_input():
    assert ob.num_frames(399) == 0 and ob.num_frames(400) == 1 and ob.num_frames(559) == 1 and ob.num_frames(560) == 2
    assert ob.num_frames(160000) == 998
    assert ob.kaldi_fbank(np.zeros(100, np.int16)).shape == (0, 80)


def test_conformer_oracle_matches_reference(conformer_golden):
    z, meta = conformer_golden
    vocab = synth.vocabulary()
    for m in meta:
        sd = synth.to_torch(synth_weights(m["wseed"]))
        cfg = oc.ConformerConfig(causal=m["streaming"])
        feat = torch.from_numpy(z[m["name"] + "/feat"])[None]
        with torch.no_grad():
            enc = oc.encode(sd, cfg, feat)
            probs = oc.ctc_probs(sd, enc)[0].numpy()
        # same library, same op order: effectively exact
        assert np.abs(enc[0].numpy() - z[m["name"] + "/enc"]).max() < 1e-5
        ids, _ = octc.best_path(probs)
        assert np.array_equal(ids, z[m["name"] + "/ids"])
        top_i = z[m["name"] + "/top_i"]
        got = np.take_along_axis(probs, top_i.astype(np.int64), axis=1)
        assert np.abs(got - z[m["name"] + "/top_p"]).max() < 5e-6     # fp32 sums run in another order on another CPU
        score, text, _ = octc.greedy_decode(probs, vocab)
        assert text == m["text"]
        assert abs(score - m["score"]) < 1e-4


def test_greedy_oracle_semantics():
    vocab = ["<blank>", "a", "b", "<space>", "<eos>"]
    probs = np.array([[0.1, 0.6, 0.3, 0, 0], [0.1, 0.6, 0.3, 0, 0], [0.9, 0.05, 0.05, 0, 0], [0.1, 0.6, 0.3, 0, 0],
                      [0.2, 0.2, 0.2, 0.4, 0], [0.3, 0.3, 0.2, 0.2, 0]], np.float32)
    score, text, toks = octc.greedy_decode(probs, vocab)
    assert toks == [1, 1, 3] and text == "aa "
    # last row: tie between id 0 and 1 -> first index (blank) wins, like np.argmax
    assert abs(score - 100.0 * np.float32((0.6 + 0.6 + 0.6 + 0.4) / 4)) < 1e-4
    assert octc.greedy_decode(np.array([[1.0, 0, 0, 0, 0]], np.float32), vocab)[:2] == (0, "")
    # streaming variant re-collapses the whole history across chunk borders
    st = octc.GreedyStream()
    st.push(probs[:2], vocab)
    s2, t2, _ = st.push(probs[2:], vocab)
    assert t2 == text and abs(s2 - score) < 1e-5
