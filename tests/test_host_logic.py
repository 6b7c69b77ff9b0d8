"""Host-side logic of the widened rows, without a GPU: the EER scalar arithmetic of evaluation.py
(s5:80-97) on oracle counts against the reference-generated goldens, and the span-offset arithmetic of
batches.py against the oracle's batch assembly (a flat numpy gather stands in for the copy kernel)."""
import os

import numpy as np
import pytest

from oracle import batch_oracle as bo
from oracle import eer_oracle as eo
from speaker_embedding_ge2e_loss_b200.batches import span_offsets
from speaker_embedding_ge2e_loss_b200.evaluation import default_thresholds, eer_from_counts

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_default_thresholds_are_the_reference_list():
    assert default_thresholds() == eo.default_thresholds() == [0.01 * i + 0.5 for i in range(50)]


def test_eer_scalar_arithmetic_matches_reference_goldens():
    z = np.load(os.path.join(GOLD, "eer_reference_vectors.npz"))
    names = [k[:-2] for k in z.files if k.endswith("_S")]
    assert len(names) >= 8
    for n in names:
        S = z[n + "_S"]
        a, o = eo.threshold_counts(S, default_thresholds())
        r = eer_from_counts(a, o, S.shape[0], S.shape[1], default_thresholds())
        assert [r.EER, r.thres, r.FAR, r.FRR] == list(z[n + "_res"])
        assert np.array_equal(np.asarray(r.far), z[n + "_far"]) and np.array_equal(np.asarray(r.frr), z[n + "_frr"])
    with pytest.raises(ValueError):
        eer_from_counts([0], [0], 1, 5, [0.5])


@pytest.mark.parametrize("name", ["s6_n4m5", "s5_n5m3_small", "s9_n8m4_odd"])
def test_span_offsets_reproduce_reference_batches(name):
    z = np.load(os.path.join(GOLD, "batch_reference_vectors.npz"))
    S, frames, mels, N, M, L, seed = (int(v) for v in z[name + "_cfg"])
    files = [z[f"{name}_file{s}"] for s in range(S)]
    flat = np.concatenate([f.astype(np.float32).reshape(-1) for f in files])            # the bank's device layout
    first = np.concatenate([[0], np.cumsum([f.shape[0] for f in files])])
    order = [int(i) for i in z[name + "_order"]]
    np.random.seed(seed)
    utt, clip = bo.draw_indices([files[s].shape[0] for s in order], M, frames, L)
    off = span_offsets(first, frames, mels, order, utt, clip, z[name + "_perm"])
    span = L * mels
    got = np.stack([flat[o:o + span] for o in off]).reshape(N * M, L, mels)
    assert got.dtype == np.float32 and np.array_equal(got, z[name + "_batch"])
    assert off.dtype == np.int64 and off.flags["C_CONTIGUOUS"] and (off % mels == 0).all()


def test_backward_envelope_query_and_refusal():
    """ge2e_b200_max_utterances (host only): the backward keeps 2 M + 2 rows of D floats (D rounded up to 4) in
    200 KB of shared memory; the Python layer refuses a larger M with a ValueError that names the limit."""
    from speaker_embedding_ge2e_loss_b200 import _lib
    h = _lib.lib()
    for D, m in [(128, 199), (256, 99), (512, 49), (768, 32), (1000, 24), (1023, 24), (1024, 24), (1, 6399)]:
        assert h.ge2e_b200_max_utterances(D) == m
        Dp = (D + 3) // 4 * 4
        assert (2 * m + 2) * Dp * 4 <= 200 * 1024 < (2 * m + 4) * Dp * 4
    assert h.ge2e_b200_max_utterances(0) == 0 and h.ge2e_b200_max_utterances(1025) == 0
    _lib.check_backward_shape(99, 256)
    with pytest.raises(ValueError, match="at most 99 utterances per speaker at D = 256"):
        _lib.check_backward_shape(100, 256)
