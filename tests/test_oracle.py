"""CPU tests of the oracle (runs everywhere, no GPU): pinned against the golden vectors generated from the
reference's own code (tools/make_golden.py, tools/make_golden_reference.py), and (CNN half, which the reference
delegates to an un-vendored detectron2) against torchvision's ResNet-50."""
import os

import pytest
import torch

from oracle import clipbert_ref as R, synth

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def weights():
    return synth.full_state_dict(42)


def _load(name):
    return torch.load(os.path.join(GOLD, name), map_location="cpu", weights_only=False)


def test_weight_generation_is_reproducible(weights):
    g = _load("transformer_retrieval.pt")
    for k, v in g["weight_checksums"].items():
        assert abs(float(weights[k].double().sum()) - v) < 1e-6 * max(1.0, abs(v)), k


def test_oracle_matches_reference_golden_retrieval(weights):
    g = _load("transformer_retrieval.pt")
    sd = {k: (v.clone().requires_grad_(True) if k.startswith("transformer.") else v) for k, v in weights.items()}
    grid = g["grid"].float().requires_grad_(True)
    rep = R.repeat_tensor_rows(grid, [g["n_ex"]] * grid.shape[0])
    seq, pooled = R.clipbert_base_model(g["ids"], rep, g["mask"], sd)
    logits = R.mlp_head(pooled, sd)
    loss = R.retrieval_loss(logits, g["labels"])
    assert torch.allclose(logits, g["logits"], atol=2e-6, rtol=1e-5)
    assert torch.allclose(loss, g["loss"], atol=2e-6)
    assert torch.allclose(pooled, g["pooled"], atol=2e-6)
    assert torch.allclose(seq[:, :2, :32], g["seq_first_rows"], atol=1e-5)
    loss.mean().backward()
    assert torch.allclose(grid.grad, g["dgrid"].float(), atol=1e-4, rtol=2e-2)        # golden stored in bf16
    for k, n in g["grad_norms"].items():
        gr = sd["transformer." + k].grad
        assert abs(float(gr.norm()) - n) < 1e-4 * max(1.0, n), k
        assert torch.allclose(gr.flatten()[:64], g["grad_slices"][k], atol=1e-6, rtol=1e-4), k


def test_oracle_matches_reference_golden_multiple_choice_and_pretraining(weights):
    g = _load("transformer_multiple_choice.pt")
    sd = dict(weights)
    sd.update(synth.transformer_state_dict(50, num_labels=1))
    with torch.no_grad():
        o = R.multiple_choice(g["ids"], R.repeat_tensor_rows(g["grid"].float(), [5, 5]), g["mask"], sd, 5, g["labels"])
    assert torch.allclose(o["logits"], g["logits"], atol=2e-6) and torch.allclose(o["loss"], g["loss"], atol=2e-6)
    g = _load("transformer_pretraining.pt")
    sd = {k: v for k, v in weights.items() if not k.startswith("transformer.classifier.")}
    sd.update({k: v for k, v in synth.transformer_state_dict(60, head="pretraining").items() if k.startswith("transformer.cls.")})
    rep = R.repeat_tensor_rows(g["grid"].float(), [g["n_ex"]] * g["grid"].shape[0])
    with torch.no_grad():
        o = R.pretraining(g["ids"], rep, g["mask"], sd, g["mlm_labels"], g["itm_labels"])
    assert torch.allclose(o["itm_scores"], g["itm_scores"], atol=2e-6)
    assert torch.allclose(o["itm_loss"], g["itm_loss"], atol=2e-6)
    assert torch.allclose(o["mlm_loss"], g["mlm_loss"], atol=1e-5)
    assert torch.allclose(o["mlm_scores"][:, :4, :64], g["mlm_scores_slice"], atol=1e-5)
    assert torch.equal(o["mlm_scores"].argmax(-1), g["mlm_argmax"])


def test_oracle_cnn_matches_its_golden(weights):
    g = _load("cnn_grid.pt")
    with torch.no_grad():
        grid96, st = R.grid_feat_backbone(synth.synth_images(1, 2, size=96, seed=21), weights, return_stages=True)
        grid224 = R.grid_feat_backbone(synth.synth_images(1, 1, size=224, seed=22), weights)
    assert grid96.shape == (1, 2, 1, 1, 768) and grid224.shape == (1, 1, 3, 3, 768)      # 224 px -> 3x3 tokens (SURVEY §0.3)
    assert torch.allclose(grid96, g["grid96"], atol=1e-4, rtol=1e-4) and torch.allclose(grid224, g["grid224"], atol=1e-4, rtol=1e-4)
    assert torch.allclose(st["res5"][:, :32], g["res5_slice"], atol=1e-4, rtol=1e-4)


def test_oracle_matches_live_reference_import(weights):
    """Second seed, against the outputs of src/modeling/modeling.py's own classes on these inputs (reference_live.pt)."""
    gold = _load("reference_live.pt")["transformer"]
    g = torch.Generator().manual_seed(123)
    grid = torch.randn(3, 2, 3, 3, 768, generator=g).abs()
    ids, mask = synth.synth_text(3, 20, seed=77)
    labels = torch.tensor([0, 1, 1])
    ref = gold["retrieval"]
    with torch.no_grad():
        got = R.video_text_retrieval(ids, grid, mask, weights, labels=labels)
    assert torch.allclose(got["logits"], ref["logits"], atol=2e-6) and torch.allclose(got["loss"], ref["loss"], atol=2e-6)
    sd = dict(weights)
    sd.update(synth.transformer_state_dict(51, num_labels=3129))
    tgt = (torch.rand(3, 3129, generator=g) > 0.99).float()
    ref = gold["sequence_classification"]
    with torch.no_grad():
        got = R.sequence_classification(ids, grid, mask, sd, tgt)
    assert torch.allclose(got["logits"], ref["logits"], atol=2e-6) and torch.allclose(got["loss"], ref["loss"], atol=2e-6)


def test_oracle_visual_token_sampling_matches_live_reference(weights):
    """Pre-training's train-mode random sampling of visual tokens (modeling.py:15-34,80-88): same numpy seed => the oracle
    keeps the same sorted subset as the reference's own ClipBertForPreTraining in train() mode (dropout 0), whose outputs are
    stored in reference_live.pt (mlm_scores as a fixed, seeded sample of its elements plus the argmax of every row)."""
    import numpy as np
    ref = _load("reference_live.pt")["transformer"]["sampling"]
    sd = {k: v for k, v in weights.items() if not k.startswith("transformer.classifier.")}
    sd.update({k: v for k, v in synth.transformer_state_dict(60, head="pretraining").items() if k.startswith("transformer.cls.")})
    g = torch.Generator().manual_seed(5)
    grid = torch.randn(2, 2, 4, 5, 768, generator=g).abs()          # 20 visual tokens, keep 7
    ids, mask = synth.synth_text(2, 12, seed=9)
    np.random.seed(1234)
    idx = R.random_sample_indices(20, 7)
    assert idx.numel() == 7 and torch.equal(idx, idx.sort()[0]) and idx.unique().numel() == 7
    np.random.seed(1234)
    with torch.no_grad():
        got = R.pretraining(ids, grid, mask, sd, pixel_random_sampling_size=7)
    assert torch.allclose(got["itm_scores"], ref["itm_scores"], atol=2e-6)
    mlm = got["mlm_scores"]
    sample = torch.randint(0, mlm.numel(), ref["mlm_sample"].shape, generator=torch.Generator().manual_seed(17))
    assert list(mlm.shape) == ref["mlm_shape"] and torch.equal(mlm.argmax(-1), ref["mlm_argmax"])
    assert torch.allclose(mlm.flatten()[sample], ref["mlm_sample"], atol=2e-5)
    # eval mode: no sampling in the reference (self.training is False) == oracle with size 0; >= seq_len keeps everything
    with torch.no_grad():
        got_eval = R.pretraining(ids, grid, mask, sd)
        got_all = R.pretraining(ids, grid, mask, sd, pixel_random_sampling_size=100)
    assert torch.allclose(got_eval["itm_scores"], ref["itm_scores_eval"], atol=2e-6)
    assert torch.equal(got_all["itm_scores"], got_eval["itm_scores"])
    assert not torch.allclose(got["itm_scores"], got_eval["itm_scores"], atol=1e-4)


def test_oracle_cnn_against_torchvision_resnet50(weights):
    """Independent cross-check of the d2 restatement: torchvision ResNet-50 with FrozenBN, stride moved to conv1
    (STRIDE_IN_1X1), weights mapped with the reference's own key map (src/utils/load_save.py:335-345)."""
    torchvision = pytest.importorskip("torchvision")
    from torchvision.ops import FrozenBatchNorm2d
    net = torchvision.models.resnet50(weights=None, norm_layer=lambda c: FrozenBatchNorm2d(c, eps=1e-5))
    for name in ("layer2", "layer3", "layer4"):
        blk = getattr(net, name)[0]
        blk.conv1.stride, blk.conv2.stride = (2, 2), (1, 1)
    p = "cnn.feature.backbone."
    sd = {}

    def put(tv_conv, tv_bn, d2):
        sd[tv_conv + ".weight"] = weights[p + d2 + ".weight"]
        for a, b in (("weight", "weight"), ("bias", "bias"), ("running_mean", "running_mean"), ("running_var", "running_var")):
            sd[tv_bn + "." + a] = weights[p + d2 + ".norm." + b]

    put("conv1", "bn1", "stem.conv1")
    for li, (name, nblocks, *_r) in enumerate(R.RESNET50_STAGES):
        for b in range(nblocks):
            t, d = "layer%d.%d" % (li + 1, b), "%s.%d" % (name, b)
            for j in (1, 2, 3):
                put("%s.conv%d" % (t, j), "%s.bn%d" % (t, j), "%s.conv%d" % (d, j))
            if b == 0:
                put(t + ".downsample.0", t + ".downsample.1", d + ".shortcut")
    missing, unexpected = net.load_state_dict(sd, strict=False)
    assert all(k.startswith("fc.") for k in missing) and not unexpected
    net.eval()
    x = synth.synth_images(1, 2, size=128, seed=3).view(2, 3, 128, 128)[:, [2, 1, 0]]
    with torch.no_grad():
        y = net.maxpool(net.relu(net.bn1(net.conv1(x))))
        y = net.layer4(net.layer3(net.layer2(net.layer1(y))))
        ref = R.resnet50_res5(x, weights)
    assert torch.allclose(y, ref, atol=1e-3, rtol=1e-4)


def test_clip_aggregation_and_repeat_rows():
    g = torch.Generator().manual_seed(5)
    logits = [torch.randn(6, 2, generator=g) for _ in range(3)]
    labels = torch.randint(0, 2, (6,), generator=g)
    lg = torch.stack(logits).permute(1, 0, 2)
    want = (torch.logsumexp(lg.reshape(6, -1), -1) - torch.logsumexp(lg[:, :, :], 1).gather(1, labels[:, None]).squeeze(1)).mean()
    assert torch.allclose(R.aggregate_clip_logits(logits, labels, "lse"), want, atol=1e-6)
    assert torch.allclose(R.aggregate_clip_logits(logits, labels, "mean"),
                          torch.nn.functional.cross_entropy(torch.stack(logits).mean(0), labels), atol=1e-6)
    x = torch.arange(12.0).view(3, 4)
    assert torch.equal(R.repeat_tensor_rows(x, [1, 1, 1]), x)
    assert torch.equal(R.repeat_tensor_rows(x, [2, 1, 3]), x[[0, 0, 1, 2, 2, 2]])
    # reference quirk kept on purpose (data_utils.py:351): counts that merely SUM to len(counts) return the input unchanged
    assert torch.equal(R.repeat_tensor_rows(x, [2, 0, 1]), x)


def test_rounding_matched_oracle_stays_close_to_fp32(weights):
    batch = synth.synth_batch(1, 2, n_ex=2, size=96, seed=3)
    with torch.no_grad():
        a = R.clipbert_forward(dict(batch), weights)["logits"]
        b = R.clipbert_forward(dict(batch), weights, rnd=R.Rounding.bf16())["logits"]
    assert float((a - b).norm() / a.norm()) < 3e-2


# ------------------------------------------------------------------------------------------------
# optimizer step (SURVEY §8 f2): oracle/adamw_ref.py against the reference's own AdamW + clip_grad_norm_
# ------------------------------------------------------------------------------------------------
def _adamw_case():
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden_adamw", os.path.join(os.path.dirname(GOLD), "..", "tools", "make_golden_adamw.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_adamw_oracle_matches_reference_golden():
    from oracle import adamw_ref as A
    gold = _load("adamw.pt")
    params, grads, groups = _adamw_case().case(gold["seed"], gold["steps"])
    for g in groups:
        g["betas"] = (0.9, 0.98)
    for max_norm in (-1.0, 2.0):
        run = gold["runs"]["max_norm_%g" % max_norm]
        traj, norms = A.run(params, grads, groups, max_norm=max_norm)
        for t in range(gold["steps"]):
            for a, b in zip(traj[t], run["traj"][t]):
                assert torch.allclose(a, b, rtol=1e-6, atol=1e-8)
        for a, b in zip(norms, run["norms"]):
            assert torch.allclose(a, b, rtol=1e-6)


def test_adamw_oracle_matches_live_reference_class():
    """Second case (seed 21, 3 steps, default betas) against the parameters the reference's own AdamW left (reference_live.pt)."""
    from oracle import adamw_ref as A
    gold = _load("reference_live.pt")["adamw"]
    params, grads, groups = _adamw_case().case(seed=gold["seed"], steps=gold["steps"])
    traj, _ = A.run(params, grads, groups)
    for a, b in zip(traj[-1], gold["params"]):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-8)
