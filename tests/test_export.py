"""SURVEY.md section 8f-4: embedding export (h5 layout of coot/trainer_retrieval.py:404-415) and checkpoint files
(nntrainer/trainer_base.py:672-715) in the reference's layouts.  CPU only."""
import os

import numpy as np
import pytest
import torch as th

from coot_videotext_b200 import export as X
from coot_videotext_b200 import h5min


def test_h5min_round_trip_of_every_supported_type(tmp_path):
    rng = np.random.default_rng(0)
    data = {"f32": rng.standard_normal((7, 384)).astype(np.float32), "f64": rng.standard_normal((3,)), "i64": np.arange(11, dtype=np.int64),
            "i32": np.arange(6, dtype=np.int32).reshape(2, 3), "key": ["v_abc", "v_d", "naïve_ü"], "scalarish": np.float32([1.5])}
    p = tmp_path / "t.h5"
    h5min.write_h5(p, data)
    raw = open(p, "rb").read()
    assert raw[:8] == b"\x89HDF\r\n\x1a\n" and int.from_bytes(raw[40:48], "little") == len(raw)  # signature, end-of-file address
    back = h5min.read_h5(p)
    assert sorted(back) == sorted(data)
    for k in ("f32", "f64", "i64", "i32", "scalarish"):
        assert back[k].dtype == np.asarray(data[k]).dtype and np.array_equal(back[k], data[k]), k
    assert [b.decode("utf8") for b in back["key"]] == data["key"]  # mart/recursive_caption_dataset.py:183 decodes bytes


def test_embedding_file_has_the_reference_layout(tmp_path):
    """Keys and contents that coot/trainer_retrieval.py:404-415 writes and mart/recursive_caption_dataset.py:160-185,
    test_embeddings_retrieval.py:21-35 read: clip_num, sent_num, key, <emb> (rows / ||row||) and <emb>_before_norm."""
    g = th.Generator().manual_seed(0)
    clip_num = [3, 1, 4]
    embs = {"vid_emb": th.randn(3, 768, generator=g), "par_emb": th.randn(3, 768, generator=g), "clip_emb": th.randn(8, 384, generator=g),
            "sent_emb": th.randn(8, 384, generator=g), "vid_context": th.randn(3, 384, generator=g), "par_context": th.randn(3, 384, generator=g)}
    path = tmp_path / "embeddings" / "embeddings_7.h5"
    X.save_embeddings(path, ["v_1", "v_22", "v_333"], clip_num, clip_num, embs, use_h5py=False)
    back = X.load_embeddings(path)
    assert set(back) == {"clip_num", "sent_num", "key"} | set(embs) | {f"{k}_before_norm" for k in embs}
    assert back["clip_num"].tolist() == clip_num and back["sent_num"].tolist() == clip_num
    assert [k.decode("utf8") for k in back["key"]] == ["v_1", "v_22", "v_333"]
    for k, v in embs.items():
        assert np.array_equal(back[f"{k}_before_norm"], v.numpy())
        ref = (v / (v * v).sum(dim=-1).sqrt().unsqueeze(-1)).numpy()  # the reference's normalisation, :397-398
        assert np.array_equal(back[k], ref)
    # the retrieval check of test_embeddings_retrieval.py runs on the stored normalised embeddings
    from oracle import retrieval_oracle as RO
    res, *_ = RO.compute_retrieval(back["clip_emb"], back["sent_emb"])
    assert 0.0 <= res["r1"] <= 1.0


def test_checkpoint_files_round_trip_with_the_reference_manager(tmp_path):
    from coot_videotext_b200.model_retrieval import RetrievalModelManager
    from tests.test_nets_cpu import golden_layout, layout, reference_managers
    mine = RetrievalModelManager(vid_feat_dim=64, text_feat_dim=96)
    X.save_checkpoint(tmp_path, 3, mine, opt_state={"optimizer": {"state": {}}, "lr_scheduler": {"step": 5}})
    assert os.path.isfile(tmp_path / "models" / "model_3.pth") and os.path.isfile(tmp_path / "models" / "optimizer_3.pth")
    other = RetrievalModelManager(vid_feat_dim=64, text_feat_dim=96)
    opt = X.load_checkpoint(tmp_path, 3, other)
    assert opt["lr_scheduler"]["step"] == 5
    for net, sd in mine.get_model_state().items():
        for k, v in sd.items():
            assert th.equal(other.get_model_state()[net][k], v)
    # the reference's own manager loads the same file (trainer_base.py:703-705): one state dict per net, each with exactly the
    # names, shapes and dtypes of the reference manager's (its load_state_dict is strict)
    ref = reference_managers()["dims_64_96"]["state"]
    saved = th.load(X.models_file(tmp_path, 3))
    assert sorted(saved) == sorted(ref)
    for net, sd in saved.items():
        assert layout(sd) == golden_layout(ref[net]), net
        for k, v in sd.items():
            assert th.equal(mine.get_model_state()[net][k], v), (net, k)
