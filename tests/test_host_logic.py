"""CPU tests of the host-side logic around the kernels: flat parameter storage, state_dict contract,
the world_size-2 gradient exchange (gloo), synthetic-workload and FLOP accounting helpers."""
import contextlib
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from util import make_cfg


def test_state_dict_keys_match_the_reference_contract():
    import clipbert_b200 as cb
    from oracle import synth
    model = cb.ClipBert(make_cfg(), detectron2_model_cfg="R-50-grid.yaml")
    sd = synth.full_state_dict(42)
    assert set(model.state_dict().keys()) == set(sd.keys())            # SURVEY.md App. B
    res = model.load_state_dict(sd)
    assert not res.missing_keys
    names = [n for n, _ in model.named_parameters()]
    assert all(n.startswith(("cnn.", "transformer.")) for n in names) and any("grid_encoder" in n for n in names)
    # d2 FREEZE_AT=2: stem + res2 frozen, res3-5 + grid_encoder + transformer trainable
    frozen = [n for n, p in model.named_parameters() if not p.requires_grad]
    assert frozen and all(("stem" in n) or ("res2" in n) for n in frozen)
    n_tr = sum(p.numel() for n, p in model.named_parameters() if p.requires_grad)
    assert abs(n_tr - 148.6e6) < 0.3e6                                   # SURVEY.md §8d allreduce payload
    assert "FREEZE_AT: 2" in model.cnn.config_file
    model.freeze_cnn_backbone()
    assert [n for n, p in model.cnn.named_parameters() if p.requires_grad] == ["grid_encoder.0.weight"]


def test_flat_group_views_grads_and_conv_layout():
    from clipbert_b200.params import FlatGroup
    lin = torch.nn.Linear(24, 40)
    conv = torch.nn.Conv2d(8, 16, 3, bias=False)
    w0, c0 = lin.weight.detach().clone(), conv.weight.detach().clone()
    fg = FlatGroup(torch.device("cpu"))
    e_l = fg.add("lin.w", lin.weight)
    fg.add("lin.b", lin.bias)
    e_c = fg.add("conv.w", conv.weight, kind="conv")
    fg.materialize()
    assert torch.equal(lin.weight, w0) and torch.equal(conv.weight, c0)            # values preserved
    # conv master is stored KRSC (channels_last): element (o, c, r, s) lives at ((o*3 + r)*3 + s)*8 + c
    flat = fg.master[e_c["offset"]: e_c["offset"] + e_c["numel"]].view(16, 3, 3, 8)
    assert torch.equal(flat.permute(0, 3, 1, 2), c0)
    assert e_l["offset"] % 64 == 0 and e_c["offset"] % 64 == 0
    # grads are views of one buffer: writing the flat buffer is visible through p.grad, in the KRSC order
    fg.grad.zero_()
    fg.grad[e_c["offset"] + 5] = 3.0                                                # (o=0, r=0, s=0, c=5)
    assert float(conv.weight.grad[0, 5, 0, 0]) == 3.0
    for prm in (lin.weight, lin.bias, conv.weight):                                 # optimizer.zero_grad(set_to_none=True)
        prm.grad = None
    fg.grad.fill_(7.0)
    fg.attach_grads()
    assert conv.weight.grad is not None and float(fg.grad.abs().sum()) == 0.0       # re-attached and zeroed
    assert fg.is_current()
    lin.weight.data = lin.weight.data.clone()
    assert not fg.is_current()


def _dp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from clipbert_b200.e2e_model import allreduce_flat
    a = torch.full((1000,), float(rank + 1))
    b = torch.arange(10.0) * (rank + 1)
    works = allreduce_flat([a, b], average=True, async_op=True)
    for w in works:
        w.wait()
    q.put((rank, float(a[0]), b.tolist()))
    dist.destroy_process_group()


def test_data_parallel_gradient_exchange_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 1000
    procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, a0, b in res:
        assert a0 == pytest.approx(1.5)                                   # mean of (1, 2)
        assert b == pytest.approx([1.5 * i for i in range(10)])


def _dp_bucket_worker(rank, world, port, q):
    """Drives ClipBert's exchange bookkeeping (hooks + allreduce_grads) over gloo with stand-in halves: only the flat gradient
    buffers and the hook attributes are touched by that code."""
    import types
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from clipbert_b200.e2e_model import ClipBert
    out = {}
    for case in ("buckets", "no_buckets", "no_hooks", "transformer_frozen"):
        m = ClipBert.__new__(ClipBert)
        tf = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.full((1000,), float(rank + 1))), _grad_ready_hook=None,
                                   _pending_backward=0)
        cnn = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.zeros(640)), _bucket_hook=None, _pending_backward=0)
        object.__setattr__(m, "transformer", tf)
        object.__setattr__(m, "cnn", cnn)
        ClipBert.enable_overlapped_allreduce(m, cnn_buckets=(case in ("buckets", "transformer_frozen")))
        assert (cnn._bucket_hook is not None) == (case in ("buckets", "transformer_frozen"))
        for step in range(2):                                   # two steps: the per-step state must reset
            tf._flat.grad.fill_(float(rank + 1) * (step + 1))
            cnn._flat.grad.zero_()
            if case in ("buckets", "no_buckets"):
                tf._grad_ready_hook(tf._flat.grad)              # end of the transformer backward
            cnn._flat.grad[256:] = torch.arange(256.0, 640.0) * (rank + 1)      # res5 + grid_encoder gradients are final
            if cnn._bucket_hook is not None:
                cnn._bucket_hook(cnn._flat.grad, 256, None)
            cnn._flat.grad[:256] = torch.arange(256.0) * (rank + 1)             # res4 / res3 gradients arrive later
            ClipBert.allreduce_grads(m)
            assert m._dp["works"] == [] and m._dp["cnn_lo"] is None and m._dp["tf_started"] is False
            out[(case, step)] = (float(tf._flat.grad[0]), float(tf._flat.grad[-1]), cnn._flat.grad.tolist())
    # gradient accumulation: two micro-steps under no_sync() + one outside = ONE exchange of the accumulated buffers
    for hooks in (True, False):
        m = ClipBert.__new__(ClipBert)
        tf = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.zeros(100)), _grad_ready_hook=None, _pending_backward=0)
        cnn = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.zeros(64)), _bucket_hook=None, _pending_backward=0)
        object.__setattr__(m, "transformer", tf)
        object.__setattr__(m, "cnn", cnn)
        if hooks:
            ClipBert.enable_overlapped_allreduce(m, cnn_buckets=True)
        n_exchanged = []
        for micro in range(3):
            ctx = ClipBert.no_sync(m) if micro < 2 else contextlib.nullcontext()
            with ctx:
                tf._flat.grad += float(rank + 1)                # this rank's micro-step gradient
                cnn._flat.grad += float(10 * (rank + 1))
                if hooks:
                    tf._grad_ready_hook(tf._flat.grad)
                    cnn._bucket_hook(cnn._flat.grad, 32, None)
                ClipBert.allreduce_grads(m)
            n_exchanged.append((float(tf._flat.grad[0]), float(cnn._flat.grad[0]), float(cnn._flat.grad[-1])))
        out[("accum", hooks)] = n_exchanged
    q.put((rank, out))
    dist.destroy_process_group()


def test_bucketed_gradient_exchange_bookkeeping_world_size_2():
    """Every element of both flat buffers is averaged exactly once per step whichever hooks fired: transformer buffer from its
    hook, CNN tail [lo:) from the mid-backward bucket hook, the rest in allreduce_grads (SURVEY §8 a23 / e)."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 137) % 1000
    procs = [ctx.Process(target=_dp_bucket_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, out in res:
        for key, val in out.items():
            if key[0] == "accum":
                local = float(rank + 1)
                assert val[0] == pytest.approx((local, 10 * local, 10 * local))            # micro-step 1: untouched local sums
                assert val[1] == pytest.approx((2 * local, 20 * local, 20 * local))        # micro-step 2: still local
                assert val[2] == pytest.approx((4.5, 45.0, 45.0))                          # last: mean over ranks of 3 micro-steps
                continue
            (case, step), (t0, t1, c) = key, val
            assert t0 == pytest.approx(1.5 * (step + 1)) and t1 == pytest.approx(1.5 * (step + 1)), (case, step)
            assert c == pytest.approx([1.5 * i for i in range(640)]), (case, step)


def test_flop_accounting_matches_baseline_md():
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    assert bench.flops_per_clip(2, 41, 1) / 1e9 == pytest.approx(69.40, abs=0.05)       # BASELINE.md §3, C2 / headline
    assert bench.flops_per_clip(2, 41, 2) / 1e9 == pytest.approx(90.49, abs=0.05)
    assert bench.flops_per_clip(1, 41, 5) / 1e9 == pytest.approx(129.61, abs=0.1)
    assert bench.flops_per_clip(2, 41, 1, backward=False) / 1e9 == pytest.approx(25.23, abs=0.05)
    assert bench.flops_per_clip(1, 521, 1, backward=False) / 1e9 == pytest.approx(107.61, abs=0.1)


def test_synthetic_text_follows_the_survey_recipe():
    from oracle import synth
    ids, mask = synth.synth_text(16, 32, seed=1)
    assert ids.shape == (16, 32) and (ids[:, 0] == 101).all()
    lens = mask.sum(1)
    assert int(lens.min()) >= 8 and int(lens.max()) <= 32
    for i in range(16):
        n = int(lens[i])
        assert int(ids[i, n - 1]) == 102 and (ids[i, n:] == 0).all() and (mask[i, :n] == 1).all()


@pytest.mark.parametrize("counts", [[1, 1, 1], [2, 1, 3], [5, 5]])
def test_forward_clips_index_plan_reproduces_the_reference_clip_loop(counts, monkeypatch):
    """ClipBert.forward_clips (SURVEY §8 f1) only re-indexes: with the model replaced by a row-wise stand-in, one batched pass
    must give exactly the tensor the reference loop builds with torch.stack (run_video_retrieval.py:388-404) - bit-exact index op."""
    import clipbert_b200 as cb
    model = cb.ClipBert(make_cfg(), detectron2_model_cfg="R-50-grid.yaml")
    n_clips, T, B = 3, 2, len(counts)
    g = torch.Generator().manual_seed(5)
    vis = torch.randn(B, n_clips * T, 3, 4, 4, generator=g)
    ids = torch.randint(0, 1000, (sum(counts), 6), generator=g)
    mask = torch.ones_like(ids)

    def fake_forward(self, batch):
        # one "logit" pair per text row from (its video's frames of this clip, its own ids): what any per-row model computes
        reps = batch["n_examples_list"]
        v = batch["visual_inputs"].flatten(1).sum(1)                                   # (units,)
        v = torch.repeat_interleave(v, torch.tensor(reps))
        t = batch["text_input_ids"].float().sum(1)
        return dict(logits=torch.stack([v * 3 + t, v - t], dim=1), loss=0)
    monkeypatch.setattr(cb.ClipBert, "forward", fake_forward)
    visr = vis.view(B, n_clips, T, 3, 4, 4)
    loop = torch.stack([model.forward(dict(visual_inputs=visr[:, c], text_input_ids=ids, text_input_mask=mask, n_examples_list=list(counts)))["logits"]
                        for c in range(n_clips)])
    out = model.forward_clips(dict(visual_inputs=vis, text_input_ids=ids, text_input_mask=mask, n_examples_list=list(counts)), n_clips)["logits"]
    assert out.shape == (n_clips, sum(counts), 2) and torch.equal(out, loop)


def test_reference_setup_e2e_optimizer_runs_unchanged_on_this_model():
    """The reference's own setup_e2e_optimizer (src/optimization/utils.py:96-161) builds its 8 parameter groups from THIS
    package's ClipBert by parameter name alone - the drop-in contract of SURVEY.md §8b. The groups it built, as parameter
    names, are stored in tests/golden/reference_helpers.json (tools/make_golden_reference.py)."""
    import json
    import clipbert_b200 as cb
    from util import make_cfg
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_helpers.json")))
    model = cb.ClipBert(make_cfg(), detectron2_model_cfg="R-50-grid.yaml", transformer_cls=cb.ClipBertForVideoTextRetrieval)
    params = dict(model.named_parameters())
    groups = [dict(g, params=[params[n] for n in g["params"]]) for g in gold["optimizer_groups"]]
    assert len(groups) == 8                                      # run_video_retrieval.py:455 indexes exactly eight
    trainable = [p for p in model.parameters() if p.requires_grad]
    grouped = [p for g in groups for p in g["params"]]
    assert len(grouped) == len(trainable) and {id(p) for p in grouped} == {id(p) for p in trainable}
    names = {id(p): n for n, p in model.named_parameters()}
    # transformer: [top decay, top no-decay, rest decay, rest no-decay] with an empty prefix -> the two "top" groups are empty
    assert not groups[0]["params"] and not groups[1]["params"]
    assert all(names[id(p)].startswith("transformer.") for p in groups[2]["params"] + groups[3]["params"])
    assert all(any(nd in names[id(p)] for nd in ("bias", "LayerNorm.bias", "LayerNorm.weight")) for p in groups[3]["params"])
    assert groups[3]["weight_decay"] == 0.0 and groups[2]["weight_decay"] == 1e-3
    # cnn: the grid_encoder is the "top" group (cnn_lr_mul_prefix), res3-5 conv weights the rest; no biases in the CNN
    assert [names[id(p)] for p in groups[4]["params"]] == ["cnn.grid_encoder.0.weight"] and not groups[5]["params"] and not groups[7]["params"]
    assert len(groups[6]["params"]) == 3 * 13 + 3 and all(".res" in names[id(p)] for p in groups[6]["params"])


def test_online_softmax_recurrence_of_the_long_sequence_attention_kernel():
    """The arithmetic of attn_tc_fwd_flash_kernel (csrc/attention_tc.cu) restated tile by tile in torch - 64-key tiles, running
    row max / sum, accumulator rescaled by exp(m_old - m_new), probabilities rounded to bf16 before the P V product, -inf mask
    beyond L, -10000 on masked text keys - against plain softmax attention. (The CUDA kernel itself is checked on a B200.)"""
    g = torch.Generator().manual_seed(0)
    for L, lt in ((69, 20), (150, 100), (521, 512), (65, 0)):
        q, k, v = (torch.randn(L, 64, generator=g).bfloat16().float() for _ in range(3))
        mask = torch.ones(lt, dtype=torch.int64)
        if lt > 4:
            mask[lt // 2:] = 0
        add = torch.cat([(1.0 - mask.float()) * -10000.0, torch.zeros(L - lt)])
        s_full = q @ k.t() * 0.125 + add[None]
        ref = torch.softmax(s_full, -1) @ v
        ref_lse = torch.logsumexp(s_full, -1)
        out = torch.zeros(L, 64)
        lse = torch.zeros(L)
        for q0 in range(0, L, 64):
            qt = torch.zeros(64, 64)
            nq = min(64, L - q0)
            qt[:nq] = q[q0:q0 + nq]
            m = torch.full((64,), float("-inf"))
            ssum = torch.zeros(64)
            o = torch.zeros(64, 64)
            for k0 in range(0, L, 64):
                kt, vt = torch.zeros(64, 64), torch.zeros(64, 64)
                nk = min(64, L - k0)
                kt[:nk], vt[:nk] = k[k0:k0 + nk], v[k0:k0 + nk]
                madd = torch.full((64,), float("-inf"))
                madd[:nk] = add[k0:k0 + nk]
                s = qt @ kt.t() * 0.125 + madd[None]
                n = torch.maximum(m, s.max(-1).values)
                c = torch.exp(m - n)
                p = torch.exp(s - n[:, None])
                ssum = ssum * c + p.sum(-1)
                o = o * c[:, None] + p.bfloat16().float() @ vt
                m = n
            out[q0:q0 + nq] = (o / ssum[:, None])[:nq]
            lse[q0:q0 + nq] = (m + torch.log(ssum))[:nq]
        assert torch.isfinite(out).all()
        assert float((out - ref).norm() / ref.norm()) < 4e-3 and float((lse - ref_lse).abs().max()) < 1e-4, (L, lt)


def _nvls_worker(rank, world, port, q):
    """The NVLS exchange path of ClipBert (symmetric-memory handles, slice offsets into the multicast mapping, communication
    stream, barriers) with the CUDA-only pieces replaced: symmetric memory by plain tensors, cb_nvls_allreduce_f32 by its
    gloo restatement (tests/ops_emulator.py), streams / events by inert objects."""
    import contextlib as cl
    import types
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import torch.distributed._symmetric_memory as symm
    import ops_emulator
    from clipbert_b200 import ops
    from clipbert_b200.e2e_model import ClipBert
    from clipbert_b200.params import FlatGroup

    class _S:
        def wait_stream(self, s):
            pass

        def wait_event(self, e):
            pass

    class _E:
        def record(self, s=None):
            pass

    for name, val in (("Stream", _S), ("Event", _E), ("current_stream", lambda *a: _S()), ("stream", lambda s: cl.nullcontext())):
        setattr(torch.cuda, name, val)
    barriers = []

    class _Handle:
        def __init__(self, t):
            self.multicast_ptr, self.rank, self.world_size = t.data_ptr(), rank, world
            ops_emulator.NVLS_BUFFERS[t.data_ptr()] = t

        def barrier(self, channel=0, timeout_ms=0):
            barriers.append(channel)
            dist.barrier()
    symm.empty = lambda *size, dtype=None, device=None: torch.empty(*size, dtype=dtype)
    symm.rendezvous = lambda t, group: _Handle(t)
    ops.nvls_allreduce = ops_emulator.nvls_allreduce
    m = ClipBert.__new__(ClipBert)
    tf = types.SimpleNamespace(_flat=None, _grad_ready_hook=None, _pending_backward=0)
    cnn = types.SimpleNamespace(_flat=None, _bucket_hook=None, _pending_backward=0)
    object.__setattr__(m, "transformer", tf)
    object.__setattr__(m, "cnn", cnn)
    ClipBert.enable_overlapped_allreduce(m, cnn_buckets=True, exchange="nvls")
    assert m._dp["max_ctas"] == 64 and m._dp["tail_ctas"] == 148      # CTA count by world size: 64 up to four ranks (r02_multi_gpu.txt)
    ClipBert.enable_overlapped_allreduce(m, cnn_buckets=True, exchange="nvls", max_ctas=8)
    assert m._dp["max_ctas"] == 8
    # the gradient buffers now come from the symmetric allocator
    tf._flat = types.SimpleNamespace(grad=FlatGroup.grad_factory(1000, "cpu"))
    cnn._flat = types.SimpleNamespace(grad=FlatGroup.grad_factory(640, "cpu"))
    assert float(tf._flat.grad.abs().sum()) == 0.0                 # zero-filled
    out = []
    for step in range(2):
        tf._flat.grad.fill_(float(rank + 1) * (step + 1))
        tf._grad_ready_hook(tf._flat.grad)
        cnn._flat.grad.zero_()
        cnn._flat.grad[256:] = torch.arange(256.0, 640.0) * (rank + 1)
        cnn._bucket_hook(cnn._flat.grad, 256, None)
        cnn._flat.grad[:256] = torch.arange(256.0) * (rank + 1)
        ClipBert.allreduce_grads(m)
        out.append((float(tf._flat.grad[0]), float(tf._flat.grad[-1]), cnn._flat.grad.tolist()))
    FlatGroup.grad_factory = None
    q.put((rank, out, len(barriers), len(m._dp["handles"])))
    dist.destroy_process_group()


def test_nvls_exchange_plumbing_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 613) % 1000
    procs = [ctx.Process(target=_nvls_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, out, n_barriers, n_handles in res:
        assert n_handles == 2 and n_barriers == 2 * 3 * 2          # one rendezvous per buffer; barrier before + after each of 3 slices, 2 steps
        for step, (t0, t1, c) in enumerate(out):
            assert t0 == pytest.approx(1.5 * (step + 1)) and t1 == pytest.approx(1.5 * (step + 1))
            assert c == pytest.approx([1.5 * i for i in range(640)])


def _bf16_wire_worker(rank, world, port, q):
    """The bf16 wire format of ClipBert's exchange (persistent bf16 shadow per buffer, slice offsets, cast -> all-reduce ->
    cast back on a side stream, joined by allreduce_grads) over gloo: cb_cast_scale / cb_cast_bf16_f32 restated in torch,
    streams / events inert."""
    import contextlib as cl
    import types
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import ops_emulator
    from clipbert_b200 import ops
    from clipbert_b200.e2e_model import ClipBert

    class _S:
        def wait_stream(self, s):
            pass

        def wait_event(self, e):
            pass

    class _E:
        def record(self, s=None):
            pass

    for name, val in (("Stream", _S), ("Event", _E), ("current_stream", lambda *a: _S()), ("stream", lambda s: cl.nullcontext())):
        setattr(torch.cuda, name, val)
    ops.cast_scale, ops.cast_bf16_f32 = ops_emulator.cast_scale, ops_emulator.cast_bf16_f32
    m = ClipBert.__new__(ClipBert)
    tf = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.zeros(1000)), _grad_ready_hook=None, _pending_backward=0)
    cnn = types.SimpleNamespace(_flat=types.SimpleNamespace(grad=torch.zeros(640)), _bucket_hook=None, _pending_backward=0)
    object.__setattr__(m, "transformer", tf)
    object.__setattr__(m, "cnn", cnn)
    ClipBert.enable_overlapped_allreduce(m, cnn_buckets=True, wire="bf16")
    out = []
    for step in range(2):
        tf._flat.grad.copy_(torch.linspace(0.1, 3.0, 1000) * (rank + 1) * (step + 1))
        tf._grad_ready_hook(tf._flat.grad)
        cnn._flat.grad.zero_()
        cnn._flat.grad[256:] = torch.arange(256.0, 640.0) * (rank + 1) / 64
        cnn._bucket_hook(cnn._flat.grad, 256, None)
        cnn._flat.grad[:256] = torch.arange(256.0) * (rank + 1) / 64
        ClipBert.allreduce_grads(m)
        assert m._dp["works"] == [] and m._dp["cnn_lo"] is None
        out.append((tf._flat.grad.clone(), cnn._flat.grad.clone()))
    assert len(m._dp["shadows"]) == 2 and all(v.dtype == torch.bfloat16 for v in m._dp["shadows"].values())
    q.put((rank, out))
    dist.destroy_process_group()


def test_bf16_wire_exchange_plumbing_world_size_2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() + 377) % 1000
    procs = [ctx.Process(target=_bf16_wire_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=180) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for _, out in res:
        for step, (t, c) in enumerate(out):
            # mean over ranks (1, 2) of values rounded to bf16 before the sum, the sum rounded once more: within 2^-8 of the fp32 mean
            want_t = torch.linspace(0.1, 3.0, 1000) * 1.5 * (step + 1)
            want_c = torch.arange(640.0) * 1.5 / 64
            assert float(((t - want_t).abs() / want_t).max()) < 2 ** -7
            assert float((c - want_c).abs().max()) <= float(want_c.max()) * 2 ** -7
            assert float((t - want_t).abs().max()) > 0.0                  # it really went through bf16


def test_input_stage_resize_size_matches_the_reference_function():
    """get_resize_size for tensors (src/datasets/data_utils.py:166-198) against what the reference function returned for the same
    sizes (tests/golden/reference_helpers.json)."""
    import json
    from clipbert_b200 import input_stage as IS
    gold = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_helpers.json")))
    for h, w, s, ref_h, ref_w in gold["resize_sizes"]:
        nh, nw = IS.get_resize_size(h, w, s)
        assert max(nh, nw) == s and min(nh, nw) == int(s * min(h, w) / max(h, w))
        assert (nh, nw) == (ref_h, ref_w)
