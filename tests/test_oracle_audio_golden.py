"""The wav2vec2 oracle against the reference's own audio path (tests/golden/wav2vec_tiny.npz, made by
tests/golden/make_golden_wav2vec.py from the reference's Wav2Vec2Model subclass and get_embedding with transformers'
feature extractor)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import wav2vec2_oracle as O  # noqa: E402
from tools import synth_audio as SA  # noqa: E402

G = np.load(os.path.join(ROOT, "tests", "golden", "wav2vec_tiny.npz"))
CFG = SA.W2V_TINY
SD = SA.make_state_dict(CFG, seed=0)


def _close(a, b, tol):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    err = np.abs(a - b).max()
    assert err <= tol * max(1.0, np.abs(b).max()), err


def test_feature_normalisation():
    _close(O.feature_normalize(G["speech"]), G["input_values"], 1e-6)


def test_conv_stack():
    _close(O.conv_stack(SD, CFG, torch.from_numpy(G["input_values"])).numpy(), G["conv"], 1e-5)


def test_hidden_states():
    S = O.seq_len_of(len(G["speech"]))
    states = O.encode(SD, CFG, torch.from_numpy(G["conv"]), S)
    assert len(states) == CFG["num_hidden_layers"] + 1 == G["hidden"].shape[0]
    _close(torch.stack(states).numpy(), G["hidden"][:, 0], 1e-5)


def test_embedding_and_window_cuts():
    emb = O.get_embedding(G["speech"], SD, CFG)
    assert emb.shape == (50, CFG["num_hidden_layers"], CFG["hidden_size"])     # 2.0077 s -> int(50.19) rows
    _close(emb.numpy(), G["emb"], 1e-5)
    ref = torch.from_numpy(G["emb"])
    np.testing.assert_array_equal(O.cut_windows(ref, 13, 0).numpy(), G["cut0"])
    np.testing.assert_array_equal(O.cut_windows(ref, 13, int(G["cut_end_start"])).numpy(), G["cut_end"])
