"""Generate tests/golden/reference_live.pt and tests/golden/reference_helpers.json by running the REFERENCE's own code.

These are the comparisons the CPU tests once made against a live import of the reference tree (CLIPBERT_REFERENCE_ROOT):
what the reference computed is stored here, so the tests run on a machine without that tree and keep comparing against it.

  reference_live.pt      transformer outputs of the reference classes (retrieval, 3129-way sequence classification,
                         pre-training with train-mode visual token sampling) and the final parameters of its AdamW
  reference_helpers.json get_resize_size, setup_e2e_optimizer's parameter groups on this package's ClipBert, the key maps of
                         convert_torchvision_ckpt_to_detectron2 / load_state_dict_with_mismatch, and the horovod calls
                         (arguments and answers, world size 2 over gloo) made by all_reduce_and_rescale_tensors / broadcast_tensors

Every input is regenerated from the seeds the tests use; run with the reference tree present:
  CLIPBERT_REFERENCE_ROOT=<reference checkout> python tools/make_golden_reference.py
"""
import ast
import json
import os
import sys
import types
import warnings

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from oracle import ref_import, synth  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
REF = ref_import.REFERENCE_ROOT
MLM_SAMPLE = 32768          # mlm_scores of the sampling case are 2 x 12 x 30522: a fixed, seeded sample of them is stored


def _ref_functions(rel, names, ns):
    """Top-level functions of one reference file, executed without importing the file (its imports need apex / horovod)."""
    path = os.path.join(REF, rel)
    tree = ast.parse(open(path).read())
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in names]
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


def mlm_sample_index(numel):
    return torch.randint(0, numel, (MLM_SAMPLE,), generator=torch.Generator().manual_seed(17))


def transformer_live(weights):
    """tests/test_oracle.py::test_oracle_matches_live_reference_import and ::test_oracle_visual_token_sampling_matches_live_reference."""
    import numpy as np
    out = {}
    g = torch.Generator().manual_seed(123)
    grid = torch.randn(3, 2, 3, 3, 768, generator=g).abs()
    ids, mask = synth.synth_text(3, 20, seed=77)
    labels = torch.tensor([0, 1, 1])
    with torch.no_grad():
        ref = ref_import.build_reference_transformer(weights)(ids, grid, mask, labels=labels)
    out["retrieval"] = dict(logits=ref["logits"], loss=ref["loss"])
    sd = dict(weights)
    sd.update(synth.transformer_state_dict(51, num_labels=3129))
    tgt = (torch.rand(3, 3129, generator=g) > 0.99).float()
    model = ref_import.build_reference_transformer(sd, "ClipBertForSequenceClassification", num_labels=3129, loss_type="bce")
    with torch.no_grad():
        ref = model(ids, grid, mask, labels=tgt)
    out["sequence_classification"] = dict(logits=ref["logits"], loss=ref["loss"])

    sd = {k: v for k, v in weights.items() if not k.startswith("transformer.classifier.")}
    sd.update({k: v for k, v in synth.transformer_state_dict(60, head="pretraining").items() if k.startswith("transformer.cls.")})
    g = torch.Generator().manual_seed(5)
    grid = torch.randn(2, 2, 4, 5, 768, generator=g).abs()
    ids, mask = synth.synth_text(2, 12, seed=9)
    model = ref_import.build_reference_transformer(sd, "ClipBertForPreTraining", hidden_dropout_prob=0.0,
                                                   attention_probs_dropout_prob=0.0, pixel_random_sampling_size=7)
    model.train()
    np.random.seed(1234)
    with torch.no_grad():
        ref = model(ids, grid, mask)
    model.eval()
    with torch.no_grad():
        ref_eval = model(ids, grid, mask)
    mlm = ref["mlm_scores"]
    out["sampling"] = dict(itm_scores=ref["itm_scores"], mlm_shape=list(mlm.shape), mlm_argmax=mlm.argmax(-1),
                           mlm_sample=mlm.flatten()[mlm_sample_index(mlm.numel())].clone(), itm_scores_eval=ref_eval["itm_scores"])
    return out


def adamw_live():
    """tests/test_oracle.py::test_adamw_oracle_matches_live_reference_class: the reference's AdamW driven as the test drives it."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_adamw", os.path.join(REF, "src", "optimization", "adamw.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    spec = importlib.util.spec_from_file_location("make_golden_adamw", os.path.join(ROOT, "tools", "make_golden_adamw.py"))
    mk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mk)
    params, grads, groups = mk.case(seed=21, steps=3)
    ps = [torch.nn.Parameter(p.clone()) for p in params]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        opt = m.AdamW([dict(params=[ps[i] for i in g["idx"]], lr=g["lr"], weight_decay=g["weight_decay"]) for g in groups], lr=1e-4)
        for gs in grads:
            for p, g_ in zip(ps, gs):
                p.grad = g_.clone()
            opt.step()
    return dict(seed=21, steps=3, params=[p.detach().clone() for p in ps])


def resize_sizes():
    """tests/test_host_logic.py::test_input_stage_resize_size_matches_the_reference_function."""
    fn = _ref_functions(os.path.join("src", "datasets", "data_utils.py"), {"get_resize_size"}, {"torch": torch})["get_resize_size"]
    cases = [(360, 640, 448), (640, 360, 448), (224, 224, 224), (37, 53, 96), (1080, 1920, 768), (500, 499, 1000)]
    return [[h, w, s] + list(fn(torch.zeros(3, h, w), s)) for h, w, s in cases]


def optimizer_groups():
    """tests/test_host_logic.py::test_reference_setup_e2e_optimizer_runs_unchanged_on_this_model: setup_e2e_optimizer's groups as
    parameter names of this package's ClipBert."""
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from src.optimization.utils import setup_e2e_optimizer
    import clipbert_b200 as cb
    from util import make_cfg
    model = cb.ClipBert(make_cfg(), detectron2_model_cfg="R-50-grid.yaml", transformer_cls=cb.ClipBertForVideoTextRetrieval)
    opts = types.SimpleNamespace(learning_rate=5e-5, weight_decay=1e-3, transformer_lr_mul=1.0, transformer_lr_mul_prefix="",
                                 cnn_learning_rate=5e-5, cnn_weight_decay=1e-3, cnn_lr_mul=1.0, cnn_lr_mul_prefix="grid_encoder",
                                 optim="adamw", betas=(0.9, 0.98))
    names = {id(p): n for n, p in model.named_parameters()}
    return [dict(params=[names[id(p)] for p in g["params"]], lr=g["lr"], weight_decay=g["weight_decay"])
            for g in setup_e2e_optimizer(model, opts).param_groups]


def load_save_maps(tmp):
    """tests/test_load_save.py::test_helpers_agree_with_the_reference_functions: which torchvision tensor lands under which
    detectron2 name (and in which order), and which keys load_state_dict_with_mismatch hands to load_state_dict."""
    import test_load_save as T
    ns = {"torch": torch, "os": os, "Dict": dict, "Any": object, "Union": object,
          "LOGGER": types.SimpleNamespace(info=lambda *a, **k: None)}
    ref = _ref_functions(os.path.join("src", "utils", "load_save.py"),
                         {"load_state_dict_with_mismatch", "convert_torchvision_ckpt_to_detectron2"}, ns)
    tv = T._tv_resnet50_state_dict()
    tagged = {k: torch.full((1,), float(i)) for i, k in enumerate(tv)}       # each value names its source key
    path = os.path.join(tmp, "tv.pth")
    torch.save(tagged, path)
    want = ref["convert_torchvision_ckpt_to_detectron2"](path)
    src = list(tv)
    key_map = [[k, src[int(v.item())]] for k, v in want["model"].items()]
    sd = {k[len("transformer."):]: v for k, v in synth.full_state_dict(7).items() if k.startswith("transformer.")}
    sd["classifier.2.weight"] = torch.zeros(7, 1536)
    sd["extra.weight"] = torch.zeros(3)
    loaded = []
    probe = T._model().transformer
    probe.load_state_dict = lambda d, strict=True: loaded.extend(d)
    ref["load_state_dict_with_mismatch"](probe, sd)
    return dict(d2_key_map=key_map, d2_matching_heuristics=want["matching_heuristics"], mismatch_loaded_keys=sorted(loaded))


def _hvd_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import clipbert_b200.compat as compat
    compat.install()
    import horovod.torch as hvd
    hvd.init(backend="gloo")
    calls = []

    def recorded(fn):
        real = getattr(hvd, fn)

        def call(t, *args, **kwargs):
            base = t.untyped_storage().nbytes() // t.element_size()
            rec = dict(fn=fn, args=list(args), kwargs=kwargs, dtype=str(t.dtype).split(".")[-1], shape=list(t.shape),
                       base_numel=base, offset=t.storage_offset(), input=t.flatten().tolist())
            r = real(t, *args, **kwargs)
            rec["output"] = t.flatten().tolist()
            calls.append(rec)
            return r
        setattr(hvd, fn, call)
    recorded("allreduce_")
    recorded("broadcast_")
    sys.path.insert(0, REF)
    from src.utils.distributed import all_reduce_and_rescale_tensors, broadcast_tensors
    # the inputs of tests/test_compat.py::_worker
    xs = [torch.full((3,), float(rank + 1)), torch.full((2, 2), float(10 * (rank + 1)))]
    all_reduce_and_rescale_tensors(xs, 1.0)
    ys = [torch.full((3,), float(rank)), torch.full((2,), float(rank) + 5)]
    broadcast_tensors(ys, 0)
    q.put((rank, calls, [x.flatten().tolist() for x in xs], [y.tolist() for y in ys]))
    torch.distributed.destroy_process_group()


def hvd_calls():
    """tests/test_compat.py::test_horovod_and_apex_stand_ins_world_size_2: the reference's helpers on top of the stand-in."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 97) % 1000
    procs = [ctx.Process(target=_hvd_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = {r: (calls, xs, ys) for r, calls, xs, ys in (q.get(timeout=180) for _ in range(2))}
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in (0, 1):                                   # what the test asserted of the helpers' results
        calls, xs, ys = res[r]
        assert xs == [[1.5] * 3, [15.0] * 4] and ys == [[0.0] * 3, [5.0] * 2], (xs, ys)
    return {str(r): res[r][0] for r in (0, 1)}


def main():
    import tempfile
    assert ref_import.available(), "set CLIPBERT_REFERENCE_ROOT to a checkout of the reference"
    weights = synth.full_state_dict(42)
    live = dict(source="reference: src/modeling/modeling.py (via oracle/ref_import.py, fp32) and src/optimization/adamw.py",
                transformer=transformer_live(weights), adamw=adamw_live())
    torch.save(live, os.path.join(OUT, "reference_live.pt"))
    with tempfile.TemporaryDirectory() as tmp:
        maps = load_save_maps(tmp)
    helpers = dict(source="reference: src/datasets/data_utils.py get_resize_size, src/optimization/utils.py setup_e2e_optimizer, "
                          "src/utils/load_save.py, src/utils/distributed.py",
                   resize_sizes=resize_sizes(), optimizer_groups=optimizer_groups(), hvd_calls=hvd_calls(), **maps)
    with open(os.path.join(OUT, "reference_helpers.json"), "w") as f:
        json.dump(helpers, f, indent=1)
        f.write("\n")
    print("wrote tests/golden/reference_live.pt, tests/golden/reference_helpers.json")


if __name__ == "__main__":
    main()
