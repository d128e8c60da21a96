"""horovod.torch / apex stand-ins (clipbert_b200/compat, SURVEY.md §8b) over gloo, world size 2, on CPU - driven also with
the calls the reference's OWN helpers (src/utils/distributed.py) made on top of the stand-ins, recorded in
tests/golden/reference_helpers.json (tools/make_golden_reference.py)."""
import json
import os
import sys

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "reference_helpers.json")


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    import clipbert_b200.compat as compat
    assert set(compat.install()) == {"horovod.torch", "apex"}
    import horovod.torch as hvd
    from apex import amp
    hvd.init(backend="gloo")
    res = dict(size=hvd.size(), rank=hvd.rank(), local_rank=hvd.local_rank())
    # --- collectives ---
    t = torch.full((5,), float(rank + 1))
    hvd.allreduce_(t)
    res["allreduce"] = t.tolist()                                            # average: 1.5
    b = torch.arange(4.0) * (rank + 1)
    hvd.broadcast_(b, 1)
    res["broadcast"] = b.tolist()                                            # rank 1's values
    g = hvd.allgather(torch.full((rank + 1, 2), float(rank)))               # uneven first dims: 1 + 2 rows
    res["allgather"] = g.tolist()
    # --- the reference's own helpers on top of the stand-in (src/utils/distributed.py:16-41,104-139): every horovod call they
    #     made, replayed on a view of a buffer of the size they used, must get the answer it got when it was recorded ---
    res["ref_calls"] = []
    for c in json.load(open(GOLD))["hvd_calls"][str(rank)]:
        n = len(c["input"])
        t = torch.zeros(c["base_numel"], dtype=getattr(torch, c["dtype"]))[c["offset"]:c["offset"] + n].view(c["shape"])
        t.copy_(torch.tensor(c["input"]).view(c["shape"]))
        getattr(hvd, c["fn"])(t, *c["args"], **c["kwargs"])
        res["ref_calls"].append((c["fn"], t.flatten().tolist(), c["output"]))
    # --- DistributedOptimizer: gradients that are views of ONE flat buffer are exchanged as one collective ---
    flat_w, flat_g = torch.zeros(10), torch.zeros(10)
    p1, p2 = torch.nn.Parameter(flat_w[:6].view(2, 3)), torch.nn.Parameter(flat_w[6:])
    p1.grad, p2.grad = flat_g[:6].view(2, 3), flat_g[6:]
    p3 = torch.nn.Parameter(torch.zeros(2))
    p3.grad = torch.zeros(2)
    from clipbert_b200.compat.horovod_torch import _grad_buffers
    assert len(_grad_buffers([p1, p2, p3])) == 2
    opt = torch.optim.SGD([p1, p2, p3], lr=1.0)
    model, opt = amp.initialize(torch.nn.Linear(1, 1), opt, opt_level="O2")
    opt = hvd.DistributedOptimizer(opt, named_parameters=[("p1", p1), ("p2", p2), ("p3", p3)], compression=hvd.Compression.none)
    hvd.broadcast_parameters({"p1": p1, "p2": p2, "p3": p3}, root_rank=0)
    flat_g.fill_(float(rank + 1))
    p3.grad.fill_(float(2 * (rank + 1)))
    with amp.scale_loss(torch.tensor(1.0), opt) as scaled:
        assert float(scaled) == 1.0
    opt.synchronize()                                                        # reference order (:432, :492)
    res["grads"] = (flat_g.tolist(), p3.grad.tolist())
    assert [id(p) for p in amp.master_params(opt)] == [id(p1), id(p2), id(p3)]
    with opt.skip_synchronize():
        opt.step()
    res["after_step"] = (flat_w.tolist(), p3.detach().tolist())
    flat_g.fill_(float(rank + 1))                                            # plain step(): synchronizes itself
    p3.grad.zero_()
    opt.step()
    res["after_step2"] = flat_w.tolist()
    # --- optimizer state broadcast (Adam moments + step) ---
    q1 = torch.nn.Parameter(torch.ones(3) * (rank + 1))
    adam = torch.optim.Adam([q1], lr=0.1 * (rank + 1))
    q1.grad = torch.ones(3) * (rank + 1)
    adam.step()
    hvd.broadcast_parameters([("q1", q1)], root_rank=0)
    hvd.broadcast_optimizer_state(adam, root_rank=0)
    res["adam"] = (q1.detach().tolist(), adam.state[q1]["exp_avg"].tolist(), adam.param_groups[0]["lr"])
    q.put((rank, res))
    torch.distributed.destroy_process_group()


def test_horovod_and_apex_stand_ins_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 411) % 1000
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = dict(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank in (0, 1):
        r = out[rank]
        assert (r["size"], r["rank"], r["local_rank"]) == (2, rank, rank)
        assert r["allreduce"] == pytest.approx([1.5] * 5)
        assert r["broadcast"] == pytest.approx([0.0, 2.0, 4.0, 6.0])
        assert r["allgather"] == [[0.0, 0.0], [1.0, 1.0], [1.0, 1.0]]
        assert [fn for fn, _, _ in r["ref_calls"]] == ["allreduce_", "broadcast_"]
        for _, got, want in r["ref_calls"]:
            assert got == pytest.approx(want)
        assert r["grads"][0] == pytest.approx([1.5] * 10) and r["grads"][1] == pytest.approx([3.0, 3.0])
        assert r["after_step"][0] == pytest.approx([-1.5] * 10) and r["after_step"][1] == pytest.approx([-3.0, -3.0])
        assert r["after_step2"] == pytest.approx([-3.0] * 10)
    assert out[0]["adam"] == out[1]["adam"] and out[1]["adam"][2] == pytest.approx(0.1)


def test_install_leaves_real_packages_alone(monkeypatch):
    import types
    sys.path.insert(0, ROOT)
    import clipbert_b200.compat as compat
    fake = types.ModuleType("horovod")
    monkeypatch.setitem(sys.modules, "horovod", fake)
    monkeypatch.setitem(sys.modules, "apex", types.ModuleType("apex"))
    assert compat.install() == []
    assert sys.modules["horovod"] is fake


def test_reference_import_lines_resolve_to_this_package(monkeypatch, tmp_path):
    """The import lines of the reference's task scripts, verbatim (run_video_qa.py:7-11, run_pretrain.py:7-8,
    e2e_model.py:7), after compat.alias_reference_modules(): the scripts can stay byte-identical. The scripts run with the
    reference root on sys.path; an empty tree of its package layout (src/__init__.py, src/modeling/) stands in for it."""
    sys.path.insert(0, ROOT)
    import clipbert_b200 as cb
    import clipbert_b200.compat as compat
    for name in ("src.modeling.e2e_model", "src.modeling.modeling", "src.modeling.grid_feat"):
        monkeypatch.setitem(sys.modules, name, sys.modules.get(name) or __import__("types").ModuleType(name))
    (tmp_path / "src" / "modeling").mkdir(parents=True)
    (tmp_path / "src" / "__init__.py").write_text("")
    monkeypatch.syspath_prepend(str(tmp_path))
    assert compat.alias_reference_modules() == ["src.modeling.e2e_model", "src.modeling.modeling", "src.modeling.grid_feat"]
    from src.modeling.modeling import (  # noqa: F401  (run_video_qa.py:7-10)
        ClipBertForSequenceClassification,
        ClipBertForMultipleChoice,
        ClipBertForRegression)
    from src.modeling.e2e_model import ClipBert                          # run_video_qa.py:11
    from src.modeling.modeling import ClipBertForPreTraining             # run_pretrain.py:7
    from src.modeling.modeling import ClipBertForVideoTextRetrieval      # run_video_retrieval.py:7
    from src.modeling.grid_feat import GridFeatBackbone                  # e2e_model.py:7
    assert ClipBert is cb.ClipBert and ClipBertForMultipleChoice is cb.ClipBertForMultipleChoice
    assert ClipBertForSequenceClassification is cb.ClipBertForSequenceClassification and ClipBertForPreTraining is cb.ClipBertForPreTraining
    assert ClipBertForVideoTextRetrieval is cb.ClipBertForVideoTextRetrieval and GridFeatBackbone is cb.GridFeatBackbone
    with pytest.raises(NotImplementedError):       # imported by the scripts, never constructed by them
        ClipBertForRegression(None)
