"""Replay buffer (host side): behaviour against the upstream Buffer where the reference tree
is present, plus self-contained invariants (slot-0 quirk, on-disk layout, logit growth)."""
import os

import numpy as np
import pytest
import torch

import ref_shim


def _fill(buf, seed, n_batches=4, B=3, K=5):
    rng = np.random.RandomState(seed)
    for i in range(n_batches):
        data = {"examples": torch.from_numpy(rng.rand(B, 3, 8, 8).astype(np.float32)),
                "logits": torch.from_numpy(rng.randn(B, K, 2, 2).astype(np.float32)),
                "labels": torch.from_numpy(rng.randint(0, K, size=(B, 8, 8)).astype(np.int64)),
                "loss": torch.from_numpy(-rng.rand(B).astype(np.float32))}
        buf.add_data(data)


def test_buffer_invariants(tmp_path, monkeypatch):
    monkeypatch.setenv("BACS_BUFFER_ROOT", str(tmp_path))
    from bacs_b200.training.buffer import Buffer
    np.random.seed(0)
    buf = Buffer(5, "all_tasks")
    buf.update_task(task_num=0, new_class_size=5)
    assert buf.is_empty()
    _fill(buf, seed=1)
    assert buf.num_seen_examples == 12 and not buf.is_empty()
    assert os.path.exists(os.path.join(tmp_path, "mem_maps", "all_tasks", "logits_0.dat"))
    # slot 0 is never written by extend (reference quirk Q12)
    assert float(np.abs(buf.dataset_map["examples"][0]).sum()) == 0.0
    assert (buf._logits_n_classes[buf._existing_indices] == 5).all()
    buf.merge_scores()
    assert np.isclose(buf.scores.sum(), 1.0)
    # growing the number of classes zero-pads the stored logits and keeps the old values
    before = np.array(buf.dataset_map["logits"][1])
    buf.update_task(task_num=1, new_class_size=7)
    after = np.array(buf.dataset_map["logits"][1])
    assert after.shape[0] == 7 and np.array_equal(after[:5], before) and float(np.abs(after[5:]).sum()) == 0.0
    out = buf.get_data(4)
    assert out["examples"].shape == (4, 3, 8, 8) and out["logits"].shape == (4, 7, 2, 2)
    assert out["n_classes"].shape == (4,) and out["task_id"] == -1


@pytest.mark.reference
@pytest.mark.skipif(not ref_shim.reference_available(),
                    reason="upstream BACS source tree not found (set BACS_REFERENCE_ROOT)")
def test_buffer_matches_reference(tmp_path, monkeypatch):
    if not hasattr(np, "Inf"):
        monkeypatch.setattr(np, "Inf", np.inf, raising=False)     # the reference predates numpy 2
    ref = ref_shim.install()
    RefBuffer = ref["training.buffer"].Buffer
    from bacs_b200.training.buffer import Buffer
    results = []
    for cls, sub in ((RefBuffer, "ref"), (Buffer, "ours")):
        root = tmp_path / sub
        root.mkdir()
        monkeypatch.setenv("BACS_BUFFER_ROOT", str(root))
        monkeypatch.setenv("BACS_REF_CWD", str(root))
        np.random.seed(123)
        buf = cls(5, "all_tasks")
        buf.update_task(task_num=0, new_class_size=5)
        _fill(buf, seed=7, n_batches=5)
        buf.merge_scores()
        np.random.seed(5)
        out = buf.get_data(3)
        results.append((buf, out))
    (rb, ro), (ob, oo) = results
    assert np.array_equal(rb._existing_indices, ob._existing_indices)
    assert np.array_equal(rb._logits_n_classes, ob._logits_n_classes)
    assert np.allclose(rb.importance_score, ob.importance_score)
    assert np.allclose(rb.balance_score, ob.balance_score)
    assert np.allclose(rb.scores, ob.scores)
    assert rb.labels == ob.labels
    for key in ("examples", "logits", "labels"):
        assert np.array_equal(np.asarray(rb.dataset_map[key][:]), np.asarray(ob.dataset_map[key][:])), key
        assert torch.equal(ro[key], oo[key]), key
    assert np.array_equal(ro["n_classes"], oo["n_classes"])
