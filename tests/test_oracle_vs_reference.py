"""CPU: the oracle against the unmodified reference's featurizer, whole-utterance Conformer forward and chunk-by-chunk
forward of every streaming model, frozen by tests/golden/make_golden.py as fixed samples of each output
(tests/golden/reference_chunks_golden.npz)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, make_audio, synth_weights
from masr_b200 import synth
from oracle import conformer as oc, fbank as ob

# The frozen outputs were computed by the reference on one CPU.  On another, torch's fp32 CPU kernels (MKL, oneDNN, ATen)
# sum in another order: the posteriors move by up to 2.5e-6 and the Conformer's caches by up to 2.2e-6 (measured with
# the kernels limited to AVX2, to baseline x86-64 and to MKL's compatible mode).  Where the oracle and the reference run
# the same ops on the same CPU they agree bit for bit.
PROB_TOL = 5e-6


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(GOLDEN, "reference_chunks_golden.npz"))


def close(z, key, got, tol):
    """``got`` (full array) against the stored sample of the reference's array ``key``: same shape, same per-frame
    argmax (posteriors), sampled entries within ``tol``."""
    got = np.asarray(got, np.float32)
    assert got.shape == tuple(z[key + "/shape"]), key
    if key + "/ids" in z.files:
        assert np.array_equal(got.reshape(-1, got.shape[-1]).argmax(1), z[key + "/ids"]), key
    err = np.abs(got.reshape(-1)[z[key + "/idx"]] - z[key + "/val"]).max()
    assert err < tol, (key, float(err))


def test_featurizer_matches(golden):
    for kind, seed, n in [("noise", 5, 20000), ("speech", 6, 33333)]:
        close(golden, f"fbank/{kind}_{seed}", ob.featurize(make_audio(kind, seed, n)), 5e-4)
    pcm = (make_audio("speech", 7, 8000) * 20000).astype(np.int16)
    close(golden, "fbank/pcm_speech_7", ob.featurize(ob.pcm_bytes_to_float32(pcm.tobytes())), 5e-4)


def featurize(kind, seed, n):
    return torch.from_numpy(ob.featurize(make_audio(kind, seed, n)))[None]


def check_attention_chunks(z, name, encode_chunk, st, feat, first_len, cache_tol):
    """Feed ``feat`` in 67-frame windows every 64 frames (the reference's ``predict_stream`` windows, the last one short
    unless ``first_len`` == 67) and compare the posteriors and both caches after every chunk."""
    nf = feat.shape[1]
    n = 0
    for i, cur in enumerate(range(0, nf - first_len + 1, 64)):
        pm = encode_chunk(feat[:, cur:min(cur + 67, nf)], st)
        close(z, f"{name}/{i}/probs", pm, PROB_TOL)
        close(z, f"{name}/{i}/att", st.att_cache, cache_tol)
        close(z, f"{name}/{i}/cnn", st.cnn_cache, cache_tol)
        n += 1
    assert f"{name}/{n}/probs/shape" not in z.files and n > 1


def test_full_and_chunk_forward_match(golden):
    sd = synth.to_torch(synth_weights(0))
    cfg = oc.ConformerConfig()
    feat = featurize("speech", 8, 16000 * 3)
    with torch.no_grad():
        close(golden, "conformer/full", oc.get_encoder_out(sd, cfg, feat), PROB_TOL)
        check_attention_chunks(golden, "conformer", lambda ch, st: oc.get_encoder_out_chunk(sd, cfg, ch, st, -16),
                               oc.ChunkState(), feat, 67, 1e-5)


def test_squeezeformer_chunk_forward_matches(golden):
    """oracle/squeezeformer.get_encoder_out_chunk against the reference's TorchScript-able chunk method, chunk by chunk
    (probabilities and both caches), including a short final chunk."""
    from oracle import squeezeformer as osq
    sd = synth.to_torch(synth.squeezeformer_state_dict(0, streaming=True))
    cfg = osq.SqueezeformerConfig(causal=True)
    with torch.no_grad():
        check_attention_chunks(golden, "squeezeformer", lambda ch, st: osq.get_encoder_out_chunk(sd, cfg, ch, st, -16),
                               osq.ChunkState(), featurize("speech", 9, 16000 * 3 + 4000), 7, 2e-5)


def test_efficient_conformer_chunk_forward_matches(golden):
    """oracle/efficient_conformer.get_encoder_out_chunk against the reference, chunk by chunk (probabilities and
    both caches), including a short final chunk."""
    from oracle import efficient_conformer as oe
    sd = synth.to_torch(synth.efficient_conformer_state_dict(0))
    cfg = oe.EfficientConfig()
    with torch.no_grad():
        check_attention_chunks(golden, "efficient", lambda ch, st: oe.get_encoder_out_chunk(sd, cfg, ch, st, -16),
                               oe.ChunkState(), featurize("speech", 13, 16000 * 3 + 4000), 7, 2e-5)


def test_deepspeech2_chunk_forward_matches(golden):
    """oracle/deepspeech2.get_encoder_out with a carried (h, c) state against the reference's
    ``get_encoder_out_chunk`` (deepspeech2/model.py:70-77), window by window."""
    from oracle import deepspeech2 as od
    sd = synth.to_torch(synth.deepspeech2_state_dict(0, streaming=True))
    cfg = od.DS2Config(bidirectional=False)
    feat = featurize("speech", 14, 16000 * 3 + 4000)
    nf = feat.shape[1]
    state = None
    n = 0
    with torch.no_grad():
        for i, cur in enumerate(range(0, nf - 7 + 1, 64)):
            pm, state = od.get_encoder_out(sd, cfg, feat[:, cur:min(cur + 67, nf)], state)
            assert pm.shape[0] == int(golden[f"deepspeech2/{i}/len"][0])
            close(golden, f"deepspeech2/{i}/probs", pm, PROB_TOL)
            close(golden, f"deepspeech2/{i}/h", state[0].reshape(-1), 2e-5)
            close(golden, f"deepspeech2/{i}/c", state[1].reshape(-1), 2e-5)
            n += 1
    assert f"deepspeech2/{n}/len" not in golden.files and n > 1
