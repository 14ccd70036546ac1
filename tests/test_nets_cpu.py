"""CPU-side checks of the host logic: parameter containers (reference state-dict names, flat storage), synthetic batches,
cycle-loss weights."""
import json
import os
from types import SimpleNamespace

import pytest
import torch as th

from coot_videotext_b200 import synthetic as syn
from coot_videotext_b200.nets import TransformerLegacyB200, entry_names
from tests.util import GOLDEN_DIR


def test_state_dict_names_match_reference_inventory():
    """SURVEY.md section 8a parameter inventory == synthetic.net_param_shapes == the container's state_dict."""
    for kind, d_in in (("local", 96), ("global", 384)):
        net = TransformerLegacyB200(kind, d_in)
        sd = net.state_dict()
        shapes = syn.net_param_shapes(kind, d_in)
        for name, shape in shapes.items():
            assert name in sd and tuple(sd[name].shape) == tuple(shape), name
        extra = set(sd) - set(shapes)
        assert extra <= {"embedding.pe", "pooler.pools.0.genpool_one"}, extra
        assert tuple(sd["embedding.pe"].shape) == (1000, 384)


def reference_managers():
    """What the reference's RetrievalModelManager reported for the shipped configs (tests/golden/make_golden_reference_meta.py)."""
    return json.load(open(os.path.join(GOLDEN_DIR, "reference_managers.json")))


def golden_layout(entries):
    """{name: (shape, dtype)} of one net's [name, shape, dtype] list in the golden file."""
    return {k: (tuple(shape), dtype) for k, shape, dtype in entries}


def layout(sd):
    return {k: (tuple(v.shape), str(v.dtype)) for k, v in sd.items()}


def _config(reads):
    """The reference RetrievalConfig as far as it was read: attributes as a namespace, indexed entries as a dict."""
    if not isinstance(reads, dict):
        return reads
    if "__items__" in reads:
        return {k: _config(v) for k, v in reads["__items__"].items()}
    return SimpleNamespace(**{k: _config(v) for k, v in reads.items()})


@pytest.mark.parametrize("yaml_name", ["anet_coot.yaml", "yc2_100m_coot.yaml", "yc2_2d3d_coot.yaml"])
def test_manager_constructed_from_the_shipped_configs_matches_the_reference_manager(yaml_name):
    """RetrievalModelManager(cfg) with the values of the reference's own RetrievalConfig objects of the three shipped experiments:
    same state-dict names / shapes / dtypes as the reference manager, same optimizer parameter groups (names, order, decay_mult / lr_mult),
    dropout taken from the config, is_autocast_enabled() reporting like nntrainer/models/model_manager_base.py:31-38."""
    from coot_videotext_b200.model_retrieval import RetrievalModelManager
    ref = reference_managers()[yaml_name]
    cfg = _config(ref["config_reads"])
    mine = RetrievalModelManager(cfg)
    ms = mine.get_model_state()
    assert list(ms) == ref["nets"]
    for net in ms:
        assert layout(ms[net]) == golden_layout(ref["state"][net]), net
    mp, mn, mf = mine.get_all_params()
    assert mn == [g[0] for g in ref["param_groups"]] and len(ref["param_groups"]) == len(mp) == len(mf)
    for (_, decay_mult, lr_mult, shape), b in zip(ref["param_groups"], mp):
        assert decay_mult == b["decay_mult"] and lr_mult == b["lr_mult"] and list(b["params"].shape) == shape
    for net in ms:
        c = cfg.model_cfgs[net]
        assert mine.net_dropout[net][0] == c.selfatn.dropout
    assert mine.is_autocast_enabled() == ref["autocast"]["train"]
    mine.set_all_models_eval()
    assert mine.is_autocast_enabled() == ref["autocast"]["eval"]


def test_state_dict_round_trips_with_the_reference_modules():
    """A checkpoint with the reference manager's state-dict layout loads into the drop-in, and the drop-in's state dict has exactly
    that layout (names, shapes, dtypes), which is what the reference's strict load_state_dict requires."""
    from coot_videotext_b200.model_retrieval import RetrievalModelManager
    ref = reference_managers()["dims_64_96"]["state"]
    g = th.Generator().manual_seed(0)
    state = {net: {k: th.randn(shape, generator=g).to(getattr(th, dtype.split(".")[-1])) for k, shape, dtype in entries}
             for net, entries in ref.items()}
    mine = RetrievalModelManager(vid_feat_dim=64, text_feat_dim=96)
    mine.set_model_state(state)  # reference checkpoint -> drop-in
    for net in state:
        for k, v in state[net].items():
            assert th.equal(mine.model_dict[net].state_dict()[k], v), (net, k)
    for net, sd in mine.get_model_state().items():  # and back
        assert layout(sd) == golden_layout(ref[net]), net


def test_flat_storage_survives_load_and_apply():
    net = TransformerLegacyB200("local", 64)
    assert net._is_flat()
    params = syn.make_net_params("local", 64, 5)
    net.load_state_dict(params)
    assert net._is_flat()
    flat = net.flat_params()
    name, shape = entry_names("local", 64)[2]
    off = net._offsets[2]
    assert th.equal(flat[off:off + 384 * 64].view(384, 64), params["input_fc.mlp.0.weight"])
    net.double().float()  # _apply re-flattens
    assert net._is_flat()
    assert th.equal(net.state_dict()["input_fc.mlp.0.weight"], params["input_fc.mlp.0.weight"])
    # breaking the views by hand is detected and repaired
    p = net._get("norm_input.gain")
    p.data = p.data.clone()
    assert not net._is_flat()
    net.flat_params()
    assert net._is_flat()


def test_default_init_follows_reference_rules():
    """nntrainer/initialization.py:51-111: truncnorm(std 0.01, +-2 std) on weights and biases, LayerNorm left at (1, 0)."""
    net = TransformerLegacyB200("global", 384)
    sd = net.state_dict()
    w = sd["tf.encoder_layers.0.self_attention_layer.sublayer.query_projection.weight"]
    b = sd["tf.encoder_layers.0.self_attention_layer.sublayer.query_projection.bias"]
    assert float(w.abs().max()) <= 0.02 + 1e-7 and 0.005 < float(w.std()) < 0.012
    assert float(b.abs().max()) <= 0.02 + 1e-7 and float(b.abs().max()) > 0
    assert th.all(sd["norm_input.gain"] == 1) and th.all(sd["norm_input.bias"] == 0)


def test_synthetic_batch_contract():
    wl = syn.WORKLOADS["tiny"]
    b = syn.make_batch(wl, 1)
    p = int(b["clip_num"].sum())
    assert b["clip_feat"].shape == (p, wl.max_frames, wl.d_vid) and b["sent_feat"].shape[0] == p
    assert b["vid_feat_mask"].dtype == th.bool and b["clip_feat_len"].dtype == th.long
    assert float(b["clip_feat"][b["clip_feat_mask"]].abs().max()) == 0.0  # zero-filled padding
    assert th.equal(b["clip_feat_mask"], th.arange(wl.max_frames)[None] >= b["clip_feat_len"][:, None])
    b2 = syn.make_batch(wl, 1)
    assert all(th.equal(b[k], b2[k]) for k in b)


def test_cycle_weights_equal_oracle():
    from coot_videotext_b200.loss_fn import cycle_weights
    from oracle import coot_oracle as O
    lens = th.tensor([3, 1, 2])
    mask = th.arange(3)[None] >= lens[:, None]
    idx = th.tensor([2, 0, 1])
    assert th.allclose(cycle_weights(mask, lens, idx), O.cyclecons_weights(~mask, lens, idx))
    assert th.allclose(cycle_weights(mask, lens, None), O.cyclecons_weights(~mask, lens, None))
