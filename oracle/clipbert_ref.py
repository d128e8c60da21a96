"""CPU oracle for the ClipBERT forward/backward hot path — TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module, and only as the checker / the CPU arm; the product path (clipbert_b200/) never does.

Pinning status
  * Transformer half (a9-a21): restated here in plain functional PyTorch fp32 and PINNED against the
    reference's own code — src/modeling/{modeling,transformers}.py imported through oracle/ref_import.py —
    by tests/test_oracle.py, against the golden vectors under tests/golden/ that tools/make_golden.py and
    tools/make_golden_reference.py generated from that import.
  * CNN half (a2-a7): the arithmetic lives in detectron2 @ ffff8ac (docker/Dockerfile:13), which is
    NOT vendored in /root/reference and not installable offline. Restated from the published d2
    algorithm (modeling/backbone/resnet.py: BasicStem, BottleneckBlock with STRIDE_IN_1X1=True;
    layers/batch_norm.py: FrozenBatchNorm2d eps=1e-5) and anchored on the reference call sites
    src/modeling/grid_feat.py:41-48,63,89-105 and src/configs/detectron2_configs/*.yaml.
    Cross-checked against torchvision.models.resnet50(norm_layer=FrozenBatchNorm2d) with the
    stride moved to conv1 (tests/test_oracle.py). The reference holds no golden vectors for this
    path (SURVEY.md §8c) => CNN parity is "unpinned" beyond that cross-check.

All functions take a flat ``sd`` dict keyed exactly like the reference state_dict (SURVEY App. B).
"""
import math

import torch
import torch.nn.functional as F

# ----------------------------------------------------------------------------------------------
# architecture constants (src/configs/base_model.json, detectron2_configs/R-50-grid.yaml)
# ----------------------------------------------------------------------------------------------
BERT_CFG = dict(
    hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
    vocab_size=30522, max_position_embeddings=512, type_vocab_size=2, layer_norm_eps=1e-12,
    hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, initializer_range=0.02,
    max_grid_row_position_embeddings=100, max_grid_col_position_embeddings=100,
    backbone_channel_in_size=2048, pad_token_id=0)

# (stage name, #blocks, bottleneck channels, out channels, first stride) — d2 build_resnet_backbone
RESNET50_STAGES = (("res2", 3, 64, 256, 1), ("res3", 4, 128, 512, 2),
                   ("res4", 6, 256, 1024, 2), ("res5", 3, 512, 2048, 2))
FROZEN_BN_EPS = 1e-5


# ----------------------------------------------------------------------------------------------
# Rounding hooks. With the defaults (identity) every function below is the plain fp32 restatement
# that is pinned against the reference. ``Rounding.bf16()`` turns the SAME functions into the
# "bf16-rounding-matched oracle" of SURVEY.md §7: values are rounded to bf16 at exactly the points
# where the B200 path stores bf16 (activations after each fused conv / linear epilogue, tensor-core
# weight operands, FrozenBN scale folded into the conv weight before rounding), all sums stay fp32.
# ----------------------------------------------------------------------------------------------
class Rounding:
    def __init__(self, act=None, weight=None, fold_bn=False, relu_masks=None):
        self.act = act or (lambda x: x)
        self.weight = weight or (lambda w: w)
        self.fold_bn = fold_bn
        # Optional {site name: bool tensor}: replace relu(z) by z * mask at that site. Gradient tests use the
        # masks of the run under test: a ReLU net's gradient is discontinuous in its activation pattern, so two
        # forwards that differ by bf16 rounding flip ~0.1 % of the units per layer and their gradients drift apart
        # by several % per layer for reasons unrelated to the backward kernels being checked.
        self.relu_masks = relu_masks or {}
        self.pool_indices = None   # optional argmax indices (F.max_pool2d layout) for the grid_encoder max-pool

    def relu(self, z, site):
        m = self.relu_masks.get(site)
        return F.relu(z) if m is None else z * m.to(z.dtype)

    @staticmethod
    def bf16():
        r = lambda x: x.to(torch.bfloat16).to(torch.float32)   # noqa: E731
        return Rounding(act=r, weight=r, fold_bn=True)


EXACT = Rounding()


# ----------------------------------------------------------------------------------------------
# CNN: GridFeatBackbone.forward  (src/modeling/grid_feat.py:89-105)
# ----------------------------------------------------------------------------------------------
def frozen_bn(x, sd, prefix):
    """d2 FrozenBatchNorm2d: y = x*scale + shift, scale = w*rsqrt(var+eps)."""
    scale = sd[prefix + "weight"] * (sd[prefix + "running_var"] + FROZEN_BN_EPS).rsqrt()
    shift = sd[prefix + "bias"] - sd[prefix + "running_mean"] * scale
    return x * scale.view(1, -1, 1, 1) + shift.view(1, -1, 1, 1)


def conv_bn(x, sd, prefix, stride=1, padding=0, rnd=EXACT):
    if rnd.fold_bn:
        n = prefix + "norm."
        scale = sd[n + "weight"] * (sd[n + "running_var"] + FROZEN_BN_EPS).rsqrt()
        shift = sd[n + "bias"] - sd[n + "running_mean"] * scale
        w = rnd.weight(sd[prefix + "weight"] * scale.view(-1, 1, 1, 1))
        return F.conv2d(x, w, None, stride=stride, padding=padding) + shift.view(1, -1, 1, 1)
    y = F.conv2d(x, sd[prefix + "weight"], None, stride=stride, padding=padding)
    return frozen_bn(y, sd, prefix + "norm.")


def basic_stem(x, sd, prefix, rnd=EXACT):
    """d2 BasicStem: conv7x7 s2 p3 -> FrozenBN -> ReLU -> maxpool 3x3 s2 p1."""
    x = rnd.act(F.relu(conv_bn(rnd.act(x), sd, prefix + "conv1.", stride=2, padding=3, rnd=rnd)))
    return F.max_pool2d(x, kernel_size=3, stride=2, padding=1)


def bottleneck_block(x, sd, prefix, stride, has_shortcut, rnd=EXACT):
    """d2 BottleneckBlock with stride_in_1x1=True (MSRA R-50)."""
    out = rnd.act(rnd.relu(conv_bn(x, sd, prefix + "conv1.", stride=stride, rnd=rnd), prefix + "conv1"))
    out = rnd.act(rnd.relu(conv_bn(out, sd, prefix + "conv2.", stride=1, padding=1, rnd=rnd), prefix + "conv2"))
    out = conv_bn(out, sd, prefix + "conv3.", rnd=rnd)
    shortcut = rnd.act(conv_bn(x, sd, prefix + "shortcut.", stride=stride, rnd=rnd)) if has_shortcut else x
    return rnd.act(rnd.relu(out + shortcut, prefix + "out"))


def resnet50_res5(x, sd, prefix="cnn.feature.backbone.", freeze_at=2, return_stages=False, rnd=EXACT):
    """feature.backbone(x)["res5"]; stem/res2 detached from autograd when freeze_at >= 2."""
    stages = {}
    x = basic_stem(x, sd, prefix + "stem.", rnd)
    if freeze_at >= 1:
        x = x.detach()
    stages["stem"] = x
    for si, (name, nblocks, _, _, stride) in enumerate(RESNET50_STAGES):
        for b in range(nblocks):
            x = bottleneck_block(x, sd, "%s%s.%d." % (prefix, name, b), stride if b == 0 else 1, b == 0, rnd)
        if freeze_at >= si + 2:
            x = x.detach()
        stages[name] = x
    return (x, stages) if return_stages else x


def grid_feat_backbone(visual_inputs, sd, prefix="cnn.", freeze_at=2, return_stages=False, rnd=EXACT):
    """GridFeatBackbone.forward: (B,T,3,H,W) RGB float -> (B,T,h,w,768).

    view -> BGR flip (grid_feat.py:92-94) -> backbone res5 -> get_conv5_features (identity,
    grid_feats/roi_heads.py:232-236) -> grid_encoder conv3x3/maxpool2/ReLU (grid_feat.py:43-48)
    -> view/permute (grid_feat.py:100-104).
    """
    bsz, n_frms, c, h, w = visual_inputs.shape
    x = visual_inputs.reshape(bsz * n_frms, c, h, w)
    x = x[:, [2, 1, 0], :, :]
    res5, stages = resnet50_res5(x, sd, prefix + "feature.backbone.", freeze_at, return_stages=True, rnd=rnd)
    g = rnd.act(F.conv2d(res5, rnd.weight(sd[prefix + "grid_encoder.0.weight"]), None, stride=1, padding=1))
    if rnd.pool_indices is not None:      # same selection as the run under test (ties / near-ties differ otherwise)
        n_, c_ = g.shape[:2]
        g = g.flatten(2).gather(2, rnd.pool_indices.flatten(2)).view(n_, c_, g.shape[2] // 2, g.shape[3] // 2)
    else:
        g = F.max_pool2d(g, kernel_size=2, stride=2)
    g = rnd.relu(g, prefix + "grid_encoder")
    nc, nh, nw = g.shape[-3:]
    g = g.view(bsz, n_frms, nc, nh, nw).permute(0, 1, 3, 4, 2)
    if return_stages:
        stages["grid"] = g
        return g, stages
    return g


def repeat_tensor_rows(raw, row_repeats):
    """src/datasets/data_utils.py:344-357."""
    if sum(row_repeats) == len(row_repeats):
        return raw
    idx = torch.tensor([i for i, r in enumerate(row_repeats) for _ in range(r)], dtype=torch.long)
    return raw.index_select(0, idx.to(raw.device))


# ----------------------------------------------------------------------------------------------
# Transformer: ClipBertBaseModel (src/modeling/modeling.py:201-238, transformers.py)
# ----------------------------------------------------------------------------------------------
def layer_norm(x, sd, prefix, eps):
    return F.layer_norm(x, (x.shape[-1],), sd[prefix + "weight"], sd[prefix + "bias"], eps)


def linear(x, sd, prefix, rnd=EXACT):
    return F.linear(x, rnd.weight(sd[prefix + "weight"]), sd[prefix + "bias"])


def bert_embeddings(input_ids, sd, prefix, eps):
    """BertEmbeddings.forward (transformers.py:172-199), token_type 0, positions 0..Lt-1."""
    lt = input_ids.shape[1]
    e = (F.embedding(input_ids, sd[prefix + "word_embeddings.weight"])
         + sd[prefix + "position_embeddings.weight"][:lt].unsqueeze(0)
         + sd[prefix + "token_type_embeddings.weight"][0].view(1, 1, -1))
    return layer_norm(e, sd, prefix + "LayerNorm.", eps)


def random_sample_indices(seq_len, num_samples=100):
    """get_random_sample_indices (modeling.py:15-34): sorted sample without replacement drawn from numpy's GLOBAL
    generator (so np.random.seed reproduces the reference's choice); all indices when num_samples >= seq_len."""
    import numpy as np
    if num_samples >= seq_len:
        return torch.arange(seq_len)
    return torch.from_numpy(np.sort(np.random.choice(seq_len, size=num_samples, replace=False))).long()


def visual_embeddings(grid, sd, prefix, eps, sample_indices=None):
    """VisualInputEmbedding.forward (modeling.py:62-101): frame mean, +row/col, [pre-training, train mode only: keep the
    visual tokens listed in sample_indices, :80-88], +type[0], LN."""
    bsz, _, hh, ww, hsz = grid.shape
    g = grid.mean(1)
    g = g + sd[prefix + "row_position_embeddings.weight"][:hh].view(1, hh, 1, hsz)
    g = g + sd[prefix + "col_position_embeddings.weight"][:ww].view(1, 1, ww, hsz)
    v = g.reshape(bsz, -1, hsz)
    if sample_indices is not None:
        v = v.index_select(1, sample_indices.to(v.device))
    v = v + sd[prefix + "token_type_embeddings.weight"][0].view(1, 1, -1)
    return layer_norm(v, sd, prefix + "LayerNorm.", eps)


def bert_layer(h, ext_mask, sd, prefix, n_heads, eps, rnd=EXACT):
    """BertLayer.forward (transformers.py:394-418) = attention + intermediate + output."""
    b, l, d = h.shape
    hd = d // n_heads
    r = rnd.act

    def split(x):
        return x.view(b, l, n_heads, hd).permute(0, 2, 1, 3)

    q = split(r(linear(h, sd, prefix + "attention.self.query.", rnd)))
    k = split(r(linear(h, sd, prefix + "attention.self.key.", rnd)))
    v = split(r(linear(h, sd, prefix + "attention.self.value.", rnd)))
    s = torch.matmul(q, k.transpose(-1, -2)) / math.sqrt(hd) + ext_mask       # :257-264
    p = torch.softmax(s, dim=-1)
    ctx = r(torch.matmul(p, v).permute(0, 2, 1, 3).reshape(b, l, d))
    a = r(layer_norm(r(linear(ctx, sd, prefix + "attention.output.dense.", rnd) + h), sd,
                     prefix + "attention.output.LayerNorm.", eps))            # :297-301
    i = r(F.gelu(linear(a, sd, prefix + "intermediate.dense.", rnd)))         # :363-366 (erf gelu)
    return r(layer_norm(r(linear(i, sd, prefix + "output.dense.", rnd) + a), sd, prefix + "output.LayerNorm.", eps))


def clipbert_base_model(text_input_ids, grid, text_mask, sd, prefix="transformer.bert.", cfg=BERT_CFG,
                        return_layers=False, rnd=EXACT, sample_indices=None):
    """ClipBertBaseModel.forward: returns (sequence_output, pooled_output)."""
    eps = cfg["layer_norm_eps"]
    te = rnd.act(bert_embeddings(text_input_ids, sd, prefix + "embeddings.", eps))
    ve = rnd.act(visual_embeddings(rnd.act(grid), sd, prefix + "visual_embeddings.", eps, sample_indices))
    mask = torch.cat([text_mask, text_mask.new_ones(ve.shape[:2])], dim=-1)      # modeling.py:217-220
    h = torch.cat([te, ve], dim=1)                                               # [text ; visual]
    ext = (1.0 - mask[:, None, None, :].to(h.dtype)) * -10000.0                  # hf get_extended_attention_mask
    layers = [h]
    for i in range(cfg["num_hidden_layers"]):
        h = bert_layer(h, ext, sd, "%sencoder.layer.%d." % (prefix, i), cfg["num_attention_heads"], eps, rnd)
        layers.append(h)
    pooled = rnd.act(torch.tanh(linear(h[:, 0], sd, prefix + "pooler.dense.", rnd)))   # transformers.py:470-476
    if return_layers:
        return h, pooled, layers
    return h, pooled


def mlp_head(pooled, sd, prefix="transformer.classifier.", rnd=EXACT):
    """nn.Sequential(Linear(768,1536), ReLU, Linear(1536,num_labels)) (modeling.py:534-539)."""
    return linear(rnd.act(rnd.relu(linear(pooled, sd, prefix + "0.", rnd), prefix + "relu")), sd, prefix + "2.", rnd)


def retrieval_loss(logits, labels, loss_type="ce", margin=0.2, sample_size=-1):
    """ClipBertForVideoTextRetrieval.calc_loss (modeling.py:560-580)."""
    if loss_type == "ce":
        return F.cross_entropy(logits.view(-1, logits.shape[-1]), labels.view(-1), reduction="none")
    scores = torch.sigmoid(logits).squeeze().contiguous().view(sample_size, -1)
    return torch.clamp(margin + scores[:, 1:] - scores[:, :1], min=0)


def video_text_retrieval(text_input_ids, grid, text_mask, sd, labels=None, loss_type="ce", margin=0.2,
                         sample_size=-1, rnd=EXACT):
    """ClipBertForVideoTextRetrieval.forward (modeling.py:543-558), eval mode (dropout off)."""
    _, pooled = clipbert_base_model(text_input_ids, grid, text_mask, sd, rnd=rnd)
    logits = mlp_head(pooled, sd, rnd=rnd)
    loss = retrieval_loss(logits, labels, loss_type, margin, sample_size) if labels is not None else 0
    return dict(logits=logits, loss=loss)


def multiple_choice(text_input_ids, grid, text_mask, sd, num_labels, labels=None, rnd=EXACT):
    """ClipBertForMultipleChoice.forward + calc_loss with loss_type 'ce' (modeling.py:403-451)."""
    _, pooled = clipbert_base_model(text_input_ids, grid, text_mask, sd, rnd=rnd)
    logits = mlp_head(pooled, sd, rnd=rnd).view(-1, num_labels)
    loss = F.cross_entropy(logits, labels.view(-1), reduction="none") if labels is not None else 0
    return dict(logits=logits, loss=loss)


def sequence_classification(text_input_ids, grid, text_mask, sd, labels=None, loss_type="bce", rnd=EXACT):
    """ClipBertForSequenceClassification.forward (modeling.py:347-384)."""
    _, pooled = clipbert_base_model(text_input_ids, grid, text_mask, sd, rnd=rnd)
    logits = mlp_head(pooled, sd, rnd=rnd)
    if labels is None:
        loss = 0
    elif loss_type == "bce":
        loss = F.binary_cross_entropy_with_logits(logits, labels, reduction="none")   # :310-316 (reduction none)
    else:
        loss = F.cross_entropy(logits, labels.view(-1), reduction="none")
    return dict(logits=logits, loss=loss)


def pretraining(text_input_ids, grid, text_mask, sd, mlm_labels=None, itm_labels=None, cfg=BERT_CFG, pixel_random_sampling_size=0,
                rnd=EXACT):
    """ClipBertForPreTraining.forward (modeling.py:254-307); MLM head on text positions only. pixel_random_sampling_size > 0
    = the train-mode visual-token sampling of pre-training (pretrain_image_text_base_resnet50_mlm_itm.json:59)."""
    idx = None
    if pixel_random_sampling_size > 0:
        idx = random_sample_indices(grid.shape[2] * grid.shape[3], pixel_random_sampling_size)
    seq, pooled = clipbert_base_model(text_input_ids, grid, text_mask, sd, rnd=rnd, sample_indices=idx)
    lt = text_mask.shape[1]
    p = "transformer.cls.predictions."
    t = F.gelu(linear(seq[:, :lt], sd, p + "transform.dense."))
    t = layer_norm(t, sd, p + "transform.LayerNorm.", cfg["layer_norm_eps"])
    scores = F.linear(t, sd["transformer.bert.embeddings.word_embeddings.weight"], sd[p + "bias"])  # tied decoder
    itm = linear(pooled, sd, "transformer.cls.seq_relationship.")
    mlm_loss = (F.cross_entropy(scores.view(-1, scores.shape[-1]), mlm_labels.view(-1), reduction="none")
                if mlm_labels is not None else 0)
    itm_loss = F.cross_entropy(itm.view(-1, 2), itm_labels.view(-1), reduction="none") if itm_labels is not None else 0
    return dict(mlm_scores=scores, mlm_loss=mlm_loss, mlm_labels=mlm_labels, itm_scores=itm, itm_loss=itm_loss,
                itm_labels=itm_labels)


# ----------------------------------------------------------------------------------------------
# ClipBert.forward + the clip loop of the task scripts
# ----------------------------------------------------------------------------------------------
def clipbert_forward(batch, sd, head="retrieval", freeze_at=2, **head_kw):
    """ClipBert.forward (src/modeling/e2e_model.py:29-39) for one clip."""
    feats = grid_feat_backbone(batch["visual_inputs"], sd, "cnn.", freeze_at, rnd=head_kw.get("rnd", EXACT))
    feats = repeat_tensor_rows(feats, batch["n_examples_list"])
    if head == "retrieval":
        return video_text_retrieval(batch["text_input_ids"], feats, batch["text_input_mask"], sd,
                                    labels=batch.get("labels"), sample_size=len(batch["n_examples_list"]), **head_kw)
    if head == "multiple_choice":
        return multiple_choice(batch["text_input_ids"], feats, batch["text_input_mask"], sd,
                               labels=batch.get("labels"), **head_kw)
    if head == "classification":
        return sequence_classification(batch["text_input_ids"], feats, batch["text_input_mask"], sd,
                                       labels=batch.get("labels"), **head_kw)
    raise ValueError(head)


def aggregate_clip_logits(logits_per_clip, labels, pool_method="lse"):
    """Clip-level score aggregation + loss (src/tasks/run_video_retrieval.py:404-422).

    logits_per_clip: list of (B', C). Returns the scalar training loss (mean over examples).
    """
    logits = torch.stack(logits_per_clip)                       # (n_clips, B', C)
    if pool_method == "mean":
        pooled = logits.mean(0)
    elif pool_method == "max":
        pooled = logits.max(0)[0]
    elif pool_method == "lse":
        lg = logits.permute(1, 0, 2).contiguous()               # (B', n_clips, C)
        out = torch.logsumexp(lg.view(lg.shape[0], -1), dim=-1, keepdim=True) - torch.logsumexp(lg, dim=1)
        return torch.gather(out, -1, labels.view(-1, 1)).mean()
    else:
        raise ValueError(pool_method)
    return F.cross_entropy(pooled, labels.view(-1), reduction="none").mean()
