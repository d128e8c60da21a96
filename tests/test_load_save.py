"""CPU tests of the checkpoint key-layout helpers (SURVEY §8 f4, clipbert_b200/load_save.py) - index/key work, so the
bar is exact equality. What the reference's own two functions (src/utils/load_save.py) do with the same inputs is stored in
tests/golden/reference_helpers.json (tools/make_golden_reference.py) and compared key for key."""
import json
import os

import pytest
import torch

from util import make_cfg

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_helpers.json")


def _model():
    import clipbert_b200 as cb
    torch.manual_seed(11)            # identical random init for every instance (keys a checkpoint skips keep it)
    return cb.ClipBert(make_cfg(), detectron2_model_cfg="R-50-grid.yaml")


def _tv_resnet50_state_dict():
    import torchvision
    torch.manual_seed(3)
    return torchvision.models.resnet50().state_dict()


def test_torchvision_checkpoint_loads_through_the_d2_key_map():
    from clipbert_b200 import load_save as LS
    tv = _tv_resnet50_state_dict()
    d2 = LS.convert_torchvision_ckpt_to_detectron2(tv)
    assert d2["matching_heuristics"] is True and set(d2) == {"model", "__author__", "matching_heuristics"}
    assert "res3.0.shortcut.norm.running_var" in d2["model"] and "stem.conv1.norm.weight" in d2["model"] and "stem.fc.weight" in d2["model"]
    model = _model()
    loaded, ignored = LS.load_detectron2_checkpoint(model.cnn, d2)
    backbone_keys = sorted(k for k in model.cnn.state_dict() if k.startswith("feature.backbone."))
    assert loaded == backbone_keys and len(loaded) == 53 * 5                      # 53 convs x (weight + 4 FrozenBN buffers)
    assert all(k.endswith("num_batches_tracked") or k.startswith("stem.fc.") for k in ignored)
    # values land in the right tensors (KCRS view of the KRSC parameter storage)
    assert torch.equal(model.cnn.state_dict()["feature.backbone.res4.2.conv2.weight"], tv["layer3.2.conv2.weight"])
    assert torch.equal(model.cnn.state_dict()["feature.backbone.res5.0.shortcut.norm.running_mean"], tv["layer4.0.downsample.1.running_mean"])
    # the same checkpoint in d2's on-disk form: {"model": {"backbone.<...>": numpy}}
    np_ck = {"model": {"backbone." + k: v.numpy() for k, v in d2["model"].items() if not k.endswith("num_batches_tracked")}}
    model2 = _model()
    loaded2, _ = LS.load_detectron2_checkpoint(model2.cnn, np_ck)
    assert loaded2 == backbone_keys
    assert torch.equal(model2.cnn.state_dict()["feature.backbone.stem.conv1.weight"], tv["conv1.weight"])
    with pytest.raises(ValueError):
        LS.load_detectron2_checkpoint(model2.cnn, {"backbone.stem.conv1.weight": torch.zeros(64, 3, 3, 3)})


def test_load_state_dict_with_mismatch_skips_foreign_and_misshapen_keys_and_round_trips():
    from clipbert_b200 import load_save as LS
    from oracle import synth
    model = _model()
    sd = synth.full_state_dict(42)
    ck = dict(sd)
    ck["transformer.classifier.2.weight"] = torch.zeros(5, 1536)              # a checkpoint trained with another num_labels
    ck["transformer.classifier.2.bias"] = torch.zeros(5)
    ck["cnn.feature.roi_heads.box_head.fc1.weight"] = torch.zeros(4, 4)       # dead d2 head
    del ck["transformer.bert.pooler.dense.bias"]
    before = model.state_dict()["transformer.classifier.2.weight"].clone()
    rep = LS.load_state_dict_with_mismatch(model, ck)
    assert rep["mismatched"] == ["transformer.classifier.2.bias", "transformer.classifier.2.weight"]
    assert rep["unexpected"] == ["cnn.feature.roi_heads.box_head.fc1.weight"] and rep["missing"] == ["transformer.bert.pooler.dense.bias"]
    assert torch.equal(model.state_dict()["transformer.classifier.2.weight"], before)
    assert torch.equal(model.state_dict()["cnn.grid_encoder.0.weight"], sd["cnn.grid_encoder.0.weight"])
    assert model.cnn._dirty and model.transformer._dirty                     # bf16 operands are re-cast on the next forward
    out = LS.export_state_dict(model)
    assert set(out) == set(sd) and all(v.is_contiguous() and v.device.type == "cpu" for v in out.values())
    assert torch.equal(out["cnn.feature.backbone.res3.1.conv2.weight"], sd["cnn.feature.backbone.res3.1.conv2.weight"])
    fresh = _model()
    rep2 = LS.load_state_dict_with_mismatch(fresh, out)
    assert not rep2["mismatched"] and not rep2["missing"] and not rep2["unexpected"]
    assert all(torch.equal(a, b) for a, b in zip(fresh.state_dict().values(), model.state_dict().values()))


def test_helpers_agree_with_the_reference_functions(tmp_path):
    from clipbert_b200 import load_save as LS
    gold = json.load(open(GOLD))
    tv = _tv_resnet50_state_dict()
    path = str(tmp_path / "tv.pth")
    torch.save(tv, path)
    got = LS.convert_torchvision_ckpt_to_detectron2(path)
    # the reference's output: these detectron2 names, in this order, each holding the torchvision tensor named beside it
    assert list(got["model"].keys()) == [d2 for d2, _ in gold["d2_key_map"]]
    assert got["matching_heuristics"] == gold["d2_matching_heuristics"]
    assert all(torch.equal(got["model"][d2], tv[src]) for d2, src in gold["d2_key_map"])
    # load_state_dict_with_mismatch: ours against the transformer the reference's function leaves (it loads exactly these keys)
    from oracle import synth
    sd = {k[len("transformer."):]: v for k, v in synth.full_state_dict(7).items() if k.startswith("transformer.")}
    sd["classifier.2.weight"] = torch.zeros(7, 1536)
    sd["extra.weight"] = torch.zeros(3)
    a, b = _model().transformer, _model().transformer
    a.load_state_dict({k: sd[k] for k in gold["mismatch_loaded_keys"]}, strict=False)
    LS.load_state_dict_with_mismatch(b, sd)
    assert all(torch.equal(x, y) for x, y in zip(a.state_dict().values(), b.state_dict().values()))


def test_clipbert_load_state_dict_is_strict_except_for_the_dead_d2_heads():
    """TrainingRestorer calls model.load_state_dict(ckpt) (src/utils/load_save.py:283-300): a wrong or partial checkpoint must
    raise, the detectron2 RPN / ROI-head keys a reference checkpoint carries must not."""
    model = _model()
    sd = {k: v.clone() for k, v in model.state_dict().items()}
    sd["cnn.feature.roi_heads.box_head.fc1.weight"] = torch.zeros(4, 4)
    sd["cnn.feature.proposal_generator.rpn_head.conv.weight"] = torch.zeros(4, 4)
    sd["cnn.feature.pixel_mean"] = torch.zeros(3, 1, 1)
    sd["cnn.feature.backbone.stem.conv1.norm.num_batches_tracked"] = torch.zeros(())
    res = model.load_state_dict(sd)                       # strict by default: accepted
    assert not res.missing_keys
    partial = dict(sd)
    del partial["transformer.bert.pooler.dense.weight"]
    with pytest.raises(RuntimeError, match="missing keys"):
        model.load_state_dict(partial)
    model.load_state_dict(partial, strict=False)          # the tolerant form stays available
    wrong = dict(sd)
    wrong["transformer.bert.encoder.layer.12.output.dense.weight"] = torch.zeros(2, 2)
    with pytest.raises(RuntimeError, match="unexpected keys"):
        model.load_state_dict(wrong)


def test_grid_feat_backbone_loads_d2_pickles_and_names_a_missing_path(tmp_path):
    """GridFeatBackbone.load_state_dict(path) (src/modeling/grid_feat.py:72-80): detectron2 .pkl checkpoints with numpy arrays
    (the MSRA R-50.pkl layout) and .pth files load through the same key map; a path that does not exist is a clear error."""
    import pickle

    from clipbert_b200 import load_save as LS
    src, dst = _model(), _model()
    with torch.no_grad():
        for p in src.cnn.parameters():
            p.add_(0.25)
    d2 = {k[len("feature."):]: v.detach().cpu().numpy() for k, v in src.cnn.state_dict().items() if k.startswith("feature.backbone.")}
    d2["roi_heads.box_head.fc1.weight"] = torch.zeros(2, 2).numpy()
    pkl = tmp_path / "R-50.pkl"
    with open(pkl, "wb") as f:
        pickle.dump({"model": d2, "__author__": "test"}, f)
    res = dst.cnn.load_state_dict(str(pkl))
    assert "roi_heads.box_head.fc1.weight" in res.unexpected_keys
    for k, v in src.cnn.state_dict().items():
        if k.startswith("feature.backbone."):
            assert torch.equal(dst.cnn.state_dict()[k], v), k
    assert all(not k.startswith("feature.backbone.") for k in res.missing_keys)       # only grid_encoder is absent from a d2 checkpoint
    with pytest.raises(FileNotFoundError, match="does not exist"):
        dst.cnn.load_state_dict(str(tmp_path / "nope.pth"))
    with pytest.raises(ValueError, match="shape mismatch"):
        dst.cnn.load_state_dict({"backbone.stem.conv1.weight": torch.zeros(1, 1, 1, 1)})
    assert LS is not None
