#!/usr/bin/env python
"""clips/sec forward+backward of the ClipBERT hot path on N B200s (one process per GPU).

  python bench.py --gpus 1 --steps 20 --warmup 5                      # this repo's sm_100a path
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...                                # the reference's CPU path (oracle port)

One "step" = one training iteration of the reference loop (src/tasks/run_video_retrieval.py:379-432)
on one synthetic batch per GPU: for each of n_clips clips ClipBert.forward (GridFeat ResNet-50 ->
12-layer cross-modal BERT -> retrieval head), LSE aggregation of the clip logits + CE loss, backward,
and (N > 1) the data-parallel gradient all-reduce. Dropout is ON (train mode, p = 0.1) as in the
reference. 1 clip = one (video, clip) unit = T frames through the CNN + n_ex sequences through BERT.

--config selects the workload (BASELINE.json `configs`; the default, "headline", is the configuration the metric string
names: 32 videos x 2 clips x 2 frames). c2: 1 clip x 2 frames; c3: 4 clips x 2 frames; c4: TGIF-QA multiple choice, 64 videos x
2 clips x 1 frame x 5 options; c5: paragraph-retrieval INFERENCE, one video of 16 clips x 1 frame against 8 captions of 512
tokens per step (CNN once per video, one BERT pass over 128 sequences of L = 521).

JSON keys beyond the base contract:
  value     clips/s with the batch already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e       same metric through the public API (ClipBert.forward on a batch dict) with HOST (pinned)
            uint8 frames / ids / masks / labels copied H2D and the loss copied D2H every step
  roofline  the tcgen05 GEMM kernel (all convs + linears, fwd/dgrad/wgrad): algorithmic FLOPs per step
            / device time of its launches (the step's cb_gemm calls replayed back to back from a CUDA
            graph on one stream right after the timed region, CUDA events around the replay), against
            MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (oracle/clipbert_ref.py, a port: kind "port") on this host's cores
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

IMAGE_MEAN = (123.675, 116.28, 103.53)


# ------------------------------------------------------------------------------------------------
# algorithmic work (BASELINE.md §3 / SURVEY.md §8d): 1 MAC = 2 FLOP, conv / GEMM / attention contractions only
# ------------------------------------------------------------------------------------------------
def flops_per_clip(T, L, n_ex, num_labels=2, size=224, backward=True):
    scale = (size / 224.0) ** 2
    C, Cf = 4.550e9 * scale, 0.786e9 * scale
    bert = 12 * (7077888 * L + 1536 * L * L)
    head = 768 * 768 + 768 * 1536 + 1536 * num_labels
    if backward:
        return 2.0 * (T * (3 * C - 2 * Cf) + 3 * n_ex * (bert + head))
    return 2.0 * (T * C + n_ex * (bert + head))


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d.get("bf16_tflops_sustained", 1464.0), hbm=d.get("hbm_gbs", 6489.9), src="measured")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback")


def _device(local_rank):
    return torch.device("cuda", local_rank)


def _pin(t):
    return t.pin_memory()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index=0):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------
# secondary roofline: the step's largest memory-bound GEMM launch against the measured HBM copy bandwidth
# ------------------------------------------------------------------------------------------------
def gemm_algorithmic_bytes(kw):
    """Bytes of every distinct operand / result tensor of one cb_gemm launch, each counted once (SURVEY §8d)."""
    m, n, k, taps = kw["m"], kw["n"], kw["k"], kw.get("ntaps", 1)
    if kw.get("mode", 0) == 1:                              # wgrad: dY [k, m], X [k, n] -> fp32 [taps, m, n]
        return 2 * k * m + 2 * k * n + 4 * m * n * taps
    b = 2 * m * k + 2 * n * k * taps + (4 if kw.get("out_fp32") else 2) * m * n
    for t in ("residual", "aux", "out2"):
        if kw.get(t) is not None:
            b += 2 * m * n
    return b


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed `ncu --set full` capture
# (profiles/r02z_ncu_full_gemm_summary.txt, profiled launch 4: the committed round-2 kernel), keyed by the launch's shape
NCU_TRAFFIC_BYTES = {(401408, 256, 64, 1, True): 257.406208e6 + 162.649600e6}


def hbm_bound_launch(ops, rec, stream, peaks, reps=20):
    cand = [kw for kw in rec if "group" not in kw and kw.get("mode", 0) != 1 and kw.get("ntaps", 1) == 1 and kw["k"] <= 128 and kw["m"] >= 4096]
    if not cand:
        return None
    kw = max(cand, key=gemm_algorithmic_bytes)
    nbytes = gemm_algorithmic_bytes(kw)
    with torch.cuda.stream(stream):
        for _ in range(3):
            ops.gemm(**kw)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ops.gemm(**kw)
        e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / reps
    gbs = nbytes / us / 1e3
    key = (kw["m"], kw["n"], kw["k"], kw.get("ntaps", 1), kw.get("residual") is not None)
    return dict(bound="hbm", kernel="cb::gemm_kernel 1x1 conv + FrozenBN shift%s + ReLU, m=%d n=%d k=%d" % (
                    " + shortcut" if kw.get("residual") is not None else "", kw["m"], kw["n"], kw["k"]),
                achieved=round(gbs, 1), peak=peaks["hbm"], unit="GB/s", frac=round(gbs / peaks["hbm"], 4),
                peak_source="%s hbm_gbs (copy bandwidth)" % peaks["src"], algorithmic_bytes=int(nbytes), us_per_launch=round(us, 2),
                traffic=NCU_TRAFFIC_BYTES.get(key), traffic_source="profiles/r02z_ncu_full_gemm_summary.txt (ncu --set full, one launch)",
                note="%d back-to-back launches of the same problem, CUDA events on the launch stream; working set %.0f MB > 126 MB L2"
                     % (reps, nbytes / 1e6))


# ------------------------------------------------------------------------------------------------
# synthetic workload
# ------------------------------------------------------------------------------------------------
CONFIGS = {          # BASELINE.json `configs` -> workload parameters (explicit flags override)
    "headline": dict(batch=32, n_clips=2, n_frm=2, txt_len=32, n_ex=1, head="retrieval", inference=False),
    "c2": dict(batch=32, n_clips=1, n_frm=2, txt_len=32, n_ex=1, head="retrieval", inference=False),
    "c3": dict(batch=32, n_clips=4, n_frm=2, txt_len=32, n_ex=1, head="retrieval", inference=False),
    "c4": dict(batch=64, n_clips=2, n_frm=1, txt_len=32, n_ex=5, head="multiple_choice", inference=False),
    "c5": dict(batch=1, n_clips=16, n_frm=1, txt_len=512, n_ex=8, head="retrieval", inference=True),
}
METRIC_TRAIN = "clips/sec fwd+bwd MSRVTT ret (ResNet50+BERT-base)"


def apply_config(args):
    for k, v in CONFIGS[args.config].items():
        if getattr(args, k, None) is None:
            setattr(args, k, v)
    args.num_classes = 5 if args.head == "multiple_choice" else 2
    return args


def workload_name(args):
    if args.inference:
        return ("paragraph retrieval inference: %d video(s)/GPU x %d clips x %d frame(s) %dx%d against %d captions of %d tokens (CNN once per "
                "video, one BERT pass over %d sequences)" % (args.batch, args.n_clips, args.n_frm, args.size, args.size, args.n_ex, args.txt_len,
                                                              args.batch * args.n_clips * args.n_ex))
    if args.head == "multiple_choice":
        return ("TGIF-QA multiple-choice train step: %d videos/GPU x %d clips x %d frame(s) %dx%d, %d options x %d-token text, LSE clip "
                "aggregation + CE over the options, dropout 0.1, grad allreduce when N>1" % (args.batch, args.n_clips, args.n_frm, args.size, args.size,
                                                                                             args.n_ex, args.txt_len))
    return ("MSRVTT retrieval train step: %d videos/GPU x %d clips x %d frames %dx%d, %d-token text, n_ex=%d, LSE clip aggregation + CE, "
            "dropout 0.1, grad allreduce when N>1" % (args.batch, args.n_clips, args.n_frm, args.size, args.size, args.txt_len, args.n_ex))


def make_host_batch(args, rank):
    from clipbert_b200 import workload as synth   # shapes / value ranges of the synthetic inputs only
    B, frames = args.batch, args.n_clips * args.n_frm
    u8 = synth.synth_images(B, frames, size=args.size, seed=42 + rank, as_uint8=True)
    ids, mask = synth.synth_text(B * args.n_ex, args.txt_len, seed=42 + rank)
    g = torch.Generator().manual_seed(1000 + rank)
    if getattr(args, "head", "retrieval") == "multiple_choice":
        labels = torch.randint(0, args.n_ex, (B,), generator=g)          # index of the right option of each video
    else:
        labels = torch.randint(0, 2, (B * args.n_ex,), generator=g)
    pin = _pin if torch.cuda.is_available() else (lambda t: t)
    return dict(visual_inputs=pin(u8), text_input_ids=pin(ids), text_input_mask=pin(mask), labels=pin(labels))


def make_optimizer(model):
    """AdamW groups as setup_e2e_optimizer builds them (src/optimization/utils.py:96-130): decay / no-decay."""
    from clipbert_b200.optim import FusedAdamW
    no_decay = ("bias", "LayerNorm.bias", "LayerNorm.weight")
    named = [(n_, p_) for n_, p_ in model.named_parameters() if p_.requires_grad]
    return FusedAdamW([dict(params=[p_ for n_, p_ in named if not any(nd in n_ for nd in no_decay)], weight_decay=1e-3),
                       dict(params=[p_ for n_, p_ in named if any(nd in n_ for nd in no_decay)], weight_decay=0.0)],
                      lr=5e-5, betas=(0.9, 0.98), model=model)


def dump_outputs(path, model, logits, loss, inference):
    """What the timed step hands its caller, as path/<name>.npy (float32): the clip logits, and for a training step the loss and
    a fixed, seeded sample of the gradients - every trainable parameter in named_parameters() order, all of its elements up to
    1024, else max(1024, numel // 32) indices drawn from torch.Generator().manual_seed(0) (about 20 MB for ClipBERT's 149 M)."""
    import numpy as np
    out = dict(logits=torch.stack(logits) if isinstance(logits, (list, tuple)) else logits)
    if not inference:
        out["loss"] = loss
        g = torch.Generator().manual_seed(0)
        parts = []
        for _, p_ in model.named_parameters():
            if not p_.requires_grad:
                continue
            flat = p_.grad.reshape(-1)
            if flat.numel() > 1024:
                flat = flat[torch.randint(0, flat.numel(), (max(1024, flat.numel() // 32),), generator=g).to(flat.device)]
            parts.append(flat.float())
        out["grads"] = torch.cat(parts)
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        np.save(os.path.join(path, name + ".npy"), v.detach().float().cpu().numpy())
    return {name: tuple(v.shape) for name, v in out.items()}


def lse_loss(logits_per_clip, labels):
    """Clip aggregation + loss of the reference loop (run_video_retrieval.py:404-422, pool_method 'lse')."""
    lg = (logits_per_clip if torch.is_tensor(logits_per_clip) else torch.stack(logits_per_clip)).permute(1, 0, 2).contiguous()
    out = torch.logsumexp(lg.view(lg.shape[0], -1), dim=-1, keepdim=True) - torch.logsumexp(lg, dim=1)
    return torch.gather(out, -1, labels.view(-1, 1)).mean()


# ------------------------------------------------------------------------------------------------
# this repo's arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    assert world == args.gpus, "launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus)
    torch.cuda.set_device(local_rank)
    dev = _device(local_rank)
    if world > 1:
        if args.nccl_ctas:      # experiment: fewer NCCL CTAs leave more SMs to the persistent GEMMs the exchange overlaps with
            os.environ.setdefault("NCCL_MAX_CTAS", str(args.nccl_ctas))
        dist.init_process_group("nccl", device_id=dev)
    import clipbert_b200 as cb
    from clipbert_b200 import ops, workload as synth
    from clipbert_b200.workload import make_cfg

    torch.manual_seed(42)
    if args.head == "multiple_choice":    # ClipBertForMultipleChoice: one logit per (video, option) row, CE over the options
        cfg = make_cfg(num_labels=args.n_ex)
        tcls = cb.ClipBertForMultipleChoice
    else:                                 # base_model.json + retrieval head (num_labels 2, CE)
        cfg = make_cfg()
        tcls = cb.ClipBertForVideoTextRetrieval
    model = cb.ClipBert(cfg, detectron2_model_cfg="R-50-grid.yaml", transformer_cls=tcls)
    model.load_state_dict(synth.cnn_state_dict(42), strict=False)     # randomised FrozenBN statistics (random-init weights)
    model = model.to(dev)
    model = model.eval() if args.inference else model.train()
    model.cnn.pixel_mean = IMAGE_MEAN     # uint8 frames in, ImageNorm fused into the stem gather
    model.cnn.stem_mode = args.stem
    model.zero_grad_in_forward = bool(args.zero_grad_in_forward) and not args.inference
    exchange = args.exchange
    if world > 1:
        if exchange == "auto":       # this library's NVLS all-reduce where the box has a multicast mapping (N = 8: 0.956 of linear against
            exchange = "nvls" if cb.ClipBert.nvls_available(device=dev) else "nccl"          # 0.920 with NCCL, profiles/r02_multi_gpu.txt)
        model.enable_overlapped_allreduce(cnn_buckets=bool(args.cnn_buckets), exchange=exchange, max_ctas=args.nvls_ctas, wire=args.wire, tail_ctas=args.nvls_tail_ctas)

    opt = None
    ops.set_pdl(args.pdl)
    if args.sm_limit:
        ops.set_sm_limit(args.sm_limit)
    ops.set_mn3d(args.mn3d)
    ops.set_occ2(args.occ2, args.occ2_gflop)
    ops.set_attention_rows48(args.attn_rows48)
    ops.set_attention_flash_pipe(args.attn_flash_pipe)
    ops.overlap_wgrad = bool(args.overlap_wgrad)
    ops.group_wgrad = int(args.group_wgrad)
    host = make_host_batch(args, rank)
    B, n_clips, T, n_ex = args.batch, args.n_clips, args.n_frm, args.n_ex
    dbuf = {k: torch.empty(v.shape, dtype=v.dtype, device=dev) for k, v in host.items()}
    loss_host = _pin(torch.zeros(1, dtype=torch.float32))
    loss_dev = torch.zeros(1, dtype=torch.float32, device=dev)
    # logits of the latest fwd_bwd (under graph replay the captured, static output of every replay), detached and cleared
    # before the capture: a pass's autograd graph or buffers kept past its step and freed inside the capture break it
    last = {}

    def h2d():
        for k in host:
            dbuf[k].copy_(host[k], non_blocking=True)

    def fwd_bwd():
        if args.inference:         # inference_retrieval (run_video_retrieval.py:629-734): CNN once per video, then the captions
            with torch.no_grad():
                grid = model.encode_clips(dbuf["visual_inputs"], n_clips)
                mb = dict(text_input_ids=dbuf["text_input_ids"], text_input_mask=dbuf["text_input_mask"], n_examples_list=[n_ex] * B)
                logits = model.forward_clips(mb, n_clips, grid=grid)["logits"]
                loss_dev.copy_(logits.float().mean().reshape(1))          # the per-step result read back by the e2e leg
            last["logits"] = logits.detach()
            return
        if args.clip_batching:     # SURVEY §8 f1: the n_clips passes of the reference loop as ONE pass over B*n_clips units
            mb = dict(visual_inputs=dbuf["visual_inputs"], text_input_ids=dbuf["text_input_ids"], text_input_mask=dbuf["text_input_mask"],
                      n_examples_list=[n_ex] * B)
            if args.head == "retrieval":
                mb["labels"] = dbuf["labels"]     # (the QA loop hands the model labels=None and computes the loss on the stacked clip logits,
                                                  # run_video_qa.py:465-501)
            logits = model.forward_clips(mb, n_clips)["logits"]
        else:                      # the reference loop as written (run_video_retrieval.py:396-401)
            vis = dbuf["visual_inputs"].view(B, n_clips, T, 3, args.size, args.size)
            logits = []
            for c in range(n_clips):
                mb = dict(visual_inputs=vis[:, c], text_input_ids=dbuf["text_input_ids"], text_input_mask=dbuf["text_input_mask"],
                          labels=dbuf["labels"] if args.head == "retrieval" else None, n_examples_list=[n_ex] * B)
                logits.append(model(mb)["logits"])
        last["logits"] = logits.detach() if torch.is_tensor(logits) else [lg.detach() for lg in logits]
        loss = cb.clip_lse_loss(logits, dbuf["labels"]) if args.fused_loss else lse_loss(logits, dbuf["labels"])
        loss.backward()
        if world > 1:
            model.allreduce_grads()       # transformer buffer already in flight since its last backward (overlaps the CNN backward)
        loss_dev.copy_(loss.detach().reshape(1))

    graph = None
    captured_launches = 0

    def step_device():
        if not model.zero_grad_in_forward:     # else the step clears its gradient buffers itself, beside the transformer forward
            model.zero_grad()
        if graph is not None:
            graph.replay()
        else:
            fwd_bwd()

    def step_e2e():
        h2d()
        step_device()
        loss_host.copy_(loss_dev, non_blocking=True)

    # End to end with the input copy pipelined the way the reference's PrefetchLoader does it (src/datasets/dataloader.py:
    # 62-121, a side stream that uploads batch i+1 while batch i computes): every step still issues one pinned-host ->
    # device copy of a full batch inside the timed region, but on a copy stream into one of two staging sets; the step then
    # waits for its own set, moves it into the graph's fixed input buffers (device-to-device, ~6 us) and runs.
    copy_stream = torch.cuda.Stream()
    staging = [{k: torch.empty_like(v) for k, v in dbuf.items()} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    pf = dict(i=0, primed=False)

    def prefetch(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[slot])          # the step that last read this staging set has copied it out
            for k in host:
                staging[slot][k].copy_(host[k], non_blocking=True)
            ready[slot].record(copy_stream)

    def step_e2e_prefetch():
        main = torch.cuda.current_stream()
        if not pf["primed"]:
            prefetch(0)
            pf["primed"], pf["i"] = True, 0
        cur = pf["i"] & 1
        prefetch(cur ^ 1)                                # next step's inputs travel while this step computes
        main.wait_event(ready[cur])
        for k in host:
            dbuf[k].copy_(staging[cur][k], non_blocking=True)
        freed[cur].record(main)
        step_device()
        loss_host.copy_(loss_dev, non_blocking=True)
        pf["i"] += 1

    h2d()
    torch.cuda.synchronize()
    # The training script builds its optimizer before the loop (run_video_retrieval.py:296-301). With FusedAdamW the bf16
    # tensor-core operands are re-emitted by the optimizer kernel after each update (the role of apex amp O2's master ->
    # model copy inside optimizer.step, :307-309), so forward + backward - the metric - does not re-cast the weights.
    # Without an optimizer attached the modules conservatively re-cast after every backward (2 extra launches per step).
    if args.optimizer and not args.recast_in_step and not args.inference:
        try:
            model.zero_grad()
            fwd_bwd()                      # both halves now own their flat buffers (the sequence tests/test_gpu_optim.py covers)
            torch.cuda.synchronize()
            opt = make_optimizer(model)
            opt._ensure_plan()
        except Exception as e:
            if rank == 0:
                print("[bench] FusedAdamW could not be attached before the loop (%s: %s); weights are re-cast inside the step"
                      % (type(e).__name__, e), file=sys.stderr)
            opt = None
    recast_attached = opt is not None
    # ---- optional whole-step CUDA graph (fwd + bwd of all clips): removes ~900 launch latencies ----
    if args.graph:
        try:
            s = torch.cuda.Stream(priority=-1)   # the dgrad chain outranks the side queue's wgrad GEMMs for free SMs
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    model.zero_grad()
                    fwd_bwd()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            model.zero_grad()
            last.clear()
            lc0 = ops.launch_count()
            with torch.cuda.graph(g, stream=s):
                fwd_bwd()
            captured_launches = ops.launch_count() - lc0
            graph = g
        except Exception as e:      # report, fall back to eager launches (still this repo's kernels)
            if rank == 0:
                print("[bench] CUDA graph capture failed (%s: %s); running eager" % (type(e).__name__, e), file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, sample_clocks=False):
        for _ in range(warmup):
            fn()
        barrier()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        if sampler:
            sampler.start()
            time.sleep(0.15)
        l0 = ops.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = ops.launch_count() - l0
        clocks = sampler.stop() if sampler else None
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, clocks

    ms_dev, launches, clocks = timed(step_device, args.steps, args.warmup, sample_clocks=True)
    e2e_mode = "serialized"
    ms_e2e = None
    if args.prefetch:
        try:
            ms_e2e, _, _ = timed(step_e2e_prefetch, args.steps, max(3, args.warmup // 2))
            e2e_mode = "prefetch"
        except Exception as e:
            if rank == 0:
                print("[bench] pipelined input copy failed (%s: %s); measuring e2e with the copy serialized" % (type(e).__name__, e),
                      file=sys.stderr)
            torch.cuda.synchronize()
            ms_e2e = None
    if ms_e2e is None:
        ms_e2e, _, _ = timed(step_e2e, args.steps, max(3, args.warmup // 2))
    if args.dump_outputs and rank == 0:      # the last timed step's results, before the untimed passes below overwrite them
        shapes = dump_outputs(args.dump_outputs, model, last["logits"], loss_dev, args.inference)
        print("[bench] outputs of the last timed step written to %s: %s" % (args.dump_outputs, shapes), file=sys.stderr)
    if graph is not None:          # kernels replayed from the captured graph do not pass through the C-ABI counter
        launches += captured_launches * args.steps

    clips_per_step = B * n_clips * world
    L = args.txt_len + (args.size // 32 // 2) ** 2
    fl_clip = flops_per_clip(T, L, n_ex, 1 if args.head == "multiple_choice" else 2, args.size, backward=not args.inference)
    peaks = load_peaks()
    value = clips_per_step / (ms_dev / args.steps / 1e3)
    e2e_value = clips_per_step / (ms_e2e / args.steps / 1e3)

    # ---- instrumented pass: device time of the step's tcgen05 GEMM launches ----
    roof = None
    cpu = None
    try:          # every rank runs the instrumented pass (it contains the collectives); rank 0 reports. Guarded: the primary
                  # metric above must reach the JSON line even if the secondary figures cannot be produced
        # Device time of the tcgen05 GEMM launches of one step: the cb_gemm descriptors of one eager step are recorded (their
        # operand tensors stay referenced), then exactly those launches are replayed back to back from a CUDA graph on ONE
        # stream (no wgrad overlap, no PDL) and timed with CUDA events around the replay. Bracketing every launch with its own
        # event pair instead made the figure depend on the host: the GPU idles between "event recorded" and "kernel enqueued".
        ops.set_pdl(0)
        ops.overlap_wgrad = False
        ops._gemm_record = []
        model.zero_grad()
        fwd_bwd()
        torch.cuda.synchronize()
        rec, ops._gemm_record = ops._gemm_record, None
        n_gemm = len(rec)
        gs = torch.cuda.Stream()
        gs.wait_stream(torch.cuda.current_stream())
        def replay(kw):
            if "group" in kw:
                ops.gemm_wgrad_group(kw["group"])
            else:
                ops.gemm(**kw)
        with torch.cuda.stream(gs):
            for kw in rec:
                replay(kw)
        torch.cuda.synchronize()
        gg = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gg, stream=gs):
            for kw in rec:
                replay(kw)
        torch.cuda.synchronize()
        gg.replay()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            gg.replay()
        g1.record()
        torch.cuda.synchronize()
        gemm_ms = g0.elapsed_time(g1) / 5
        # ---- the largest HBM-bound launch of the step on its own (a 1x1 conv: K <= 128, far below the ~225 FLOP/B ridge) ----
        try:
            hbm_roof = hbm_bound_launch(ops, rec, gs, peaks)
        except Exception as e:          # never lose the bench line over the secondary figure
            hbm_roof = dict(error="%s: %s" % (type(e).__name__, e))
        del gg, rec
        ops.set_pdl(args.pdl)
        ops.overlap_wgrad = bool(args.overlap_wgrad)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        model.zero_grad()
        torch.cuda.synchronize()
        e0.record()
        fwd_bwd()
        e1.record()
        torch.cuda.synchronize()
        eager_ms = e0.elapsed_time(e1)
        algo_tf = fl_clip * B * n_clips / 1e12
        achieved = algo_tf / (gemm_ms / 1e3)
        roof = dict(bound="tensor", kernel="cb::gemm_kernel<BN,MODE> (tcgen05, all convs + linears fwd/dgrad/wgrad)",
                    achieved=round(achieved, 2), peak=peaks["tflops"], unit="TFLOP/s", frac=round(achieved / peaks["tflops"], 4),
                    peak_source="%s bf16_tflops_sustained" % peaks["src"], traffic=None, launches_per_step=n_gemm,
                    gemm_ms_per_step=round(gemm_ms, 3), eager_step_ms=round(eager_ms, 3),
                    gemm_share_of_step=round(gemm_ms / (ms_dev / args.steps), 3),
                    note="gemm_ms_per_step = the step's GEMM launches replayed back to back on one stream; gemm_share_of_step divides it by the "
                         "timed (two-stream) step, so wgrad/dgrad overlap can push it towards or past 1",
                    whole_step_frac=round((algo_tf * world / (ms_dev / args.steps / 1e3)) / (peaks["tflops"] * world), 4),
                    hbm_bound_launch=hbm_roof)
    except Exception as e:
        if rank == 0:
            print("[bench] roofline pass failed (%s: %s)" % (type(e).__name__, e), file=sys.stderr)
        roof = dict(bound="tensor", error="%s: %s" % (type(e).__name__, e), achieved=None, peak=peaks["tflops"], unit="TFLOP/s", frac=None,
                    traffic=None, whole_step_frac=round((fl_clip * B * n_clips / 1e12 / (ms_dev / args.steps / 1e3)) / peaks["tflops"], 4))
        ops._gemm_record = None
        ops.set_pdl(args.pdl)
        ops.overlap_wgrad = bool(args.overlap_wgrad)
        try:
            torch.cuda.synchronize()
        except Exception:
            pass
    # Ranks > 0 are done: nothing below is collective. They leave with os._exit after a last barrier - tearing the NCCL process
    # group down while CUDA graphs that captured its kernels are alive hung the run (seen at N = 2), and nothing needs cleanup.
    if world > 1:
        barrier()
        if rank != 0:
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)
    try:          # rank 0 at N = 1 only (the contract's cpu_baseline leg); never at the cost of the bench line
        cpu = None if (args.no_cpu or rank != 0 or world > 1 or args.config not in ("headline", "c2", "c3")) else cpu_baseline(args)
    except Exception as e:
        print("[bench] cpu_baseline failed (%s: %s)" % (type(e).__name__, e), file=sys.stderr)
        cpu = None
    # ---- informational: the fused optimizer step that follows fwd+bwd in training (not part of the metric) ----
    opt_info = None
    if args.optimizer and world == 1 and not args.inference:
      try:
        named = [(n_, p_) for n_, p_ in model.named_parameters() if p_.requires_grad]
        if opt is None:
            opt = make_optimizer(model)
        for _ in range(min(3, args.opt_steps)):
            opt.clip_grad_norm(1.0)
            opt.step(zero_grad=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.opt_steps):
            opt.clip_grad_norm(1.0)
            opt.step(zero_grad=True)
        e1.record()
        torch.cuda.synchronize()
        opt_ms = e0.elapsed_time(e1) / args.opt_steps
        n_el = sum(p_.numel() for _, p_ in named)
        opt_info = dict(ms_per_step=round(opt_ms, 4), params=n_el, gbytes_per_s=round(n_el * 38.0 / opt_ms / 1e6, 1),
                        note="clip_grad_norm + AdamW + zero_grad + bf16 operand emission, 3 launches per flat buffer; 38 B per parameter")
      except Exception as e:
        print("[bench] fused optimizer timing failed (%s: %s)" % (type(e).__name__, e), file=sys.stderr)
        opt_info = None

    if rank == 0:
        metric = METRIC_TRAIN if args.config in ("headline", "c2", "c3") else (
            "clips/sec inference paragraph retrieval (ResNet50+BERT-base)" if args.inference else "clips/sec fwd+bwd TGIF-QA multiple choice (ResNet50+BERT-base)")
        out = dict(metric=metric, value=round(value, 2), unit="clips/s", n_gpus=world,
                   steps=args.steps, warmup=args.warmup, ms_per_step=round(ms_dev / args.steps, 4), higher_is_better=True,
                   scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                   config=dict(workload=workload_name(args), name=args.config,
                               clips_per_step_per_gpu=B * n_clips, seq_len=L, parallelism="dp%d" % world,
                               l2="per-step working set (activations + 149 M-parameter operands, > 2 GB) >> 126 MB L2; no explicit flush",
                               cuda_graph=graph is not None, clip_batching=bool(args.clip_batching), pdl=int(args.pdl), mn3d=bool(args.mn3d), group_wgrad=int(args.group_wgrad), occ2=[args.occ2, args.occ2_gflop], overlap_wgrad=bool(args.overlap_wgrad), stem=args.stem,
                               fused_loss=bool(args.fused_loss), zero_grad_in_forward=bool(model.zero_grad_in_forward), attn_rows48=bool(args.attn_rows48), attn_flash_pipe=bool(args.attn_flash_pipe), cnn_buckets=bool(args.cnn_buckets), exchange=exchange, wire=args.wire, sm_limit=args.sm_limit, nccl_ctas=args.nccl_ctas,
                               weight_recast="in the optimizer step (FusedAdamW attached before the loop emits the bf16 operands)" if recast_attached else "inside every step (no optimizer attached)",
                               gflop_per_clip=round(fl_clip / 1e9, 2)),
                   e2e=dict(value=round(e2e_value, 2), unit="clips/s", ms_per_step=round(ms_e2e / args.steps, 4),
                            h2d_bytes_per_step=int(sum(v.numel() * v.element_size() for v in host.values())), d2h_bytes_per_step=4,
                            input_copy=("copy stream, batch i+1 uploaded while batch i computes (the reference's PrefetchLoader)"
                                        if e2e_mode == "prefetch" else "on the compute stream before each step")),
                   gpu_launches=int(launches), gpu_launches_per_step=int(launches // args.steps), clocks=clocks, roofline=roof,
                   cpu_baseline=cpu, fused_optimizer=opt_info)
        print(json.dumps(out))
    if world > 1:          # see above: no NCCL teardown with live captured graphs
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores
# ------------------------------------------------------------------------------------------------
def _cpu_step(sd, batch, n_clips, T, size):
    from oracle import clipbert_ref as R
    B = batch["visual_inputs"].shape[0]
    vis = batch["visual_inputs"].view(B, n_clips, T, 3, size, size)
    logits = []
    for c in range(n_clips):
        mb = dict(batch, visual_inputs=vis[:, c])
        logits.append(R.clipbert_forward(mb, sd)["logits"])
    loss = R.aggregate_clip_logits(logits, batch["labels"], "lse")
    loss.backward()
    return float(loss.detach())


def host_threads():
    """Threads this process can really use: affinity mask capped by the cgroup CPU quota (a container
    that sees 128 logical CPUs but is limited to a few cores collapses under 128 OpenMP threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = min(n, max(1, int(int(q[0]) / int(q[1]))))
    except Exception:
        pass
    return max(1, min(n, int(os.environ.get("CB_CPU_THREADS", 64))))


def _cpu_setup(args, b):
    from oracle import synth
    torch.set_num_threads(host_threads())
    sd = synth.full_state_dict(42)
    for k, v in sd.items():
        if k.endswith((".weight", ".bias")) and ".norm." not in k and not k.startswith(("cnn.feature.backbone.stem", "cnn.feature.backbone.res2")):
            v.requires_grad_(True)
    batch = synth.synth_batch(b, args.n_clips * args.n_frm, n_ex=args.n_ex, size=args.size, max_len=args.txt_len)
    return sd, batch


def cpu_baseline(args):
    """Bounded sample (~10-30 s) of the same workload on the host cores: fp32 eager PyTorch, all threads."""
    b = args.cpu_batch
    sd, batch = _cpu_setup(args, b)
    _cpu_step(sd, batch, args.n_clips, args.n_frm, args.size)          # warm-up
    best = 1e30
    for _ in range(2):
        t0 = time.time()
        _cpu_step(sd, batch, args.n_clips, args.n_frm, args.size)
        best = min(best, time.time() - t0)
    return dict(value=round(b * args.n_clips / best, 3), unit="clips/s", cores=torch.get_num_threads(), kind="port",
                sample="%d videos x %d clips x %d frames fwd+bwd, fp32, best of 2 after 1 warm-up (%.2f s/step)" % (b, args.n_clips, args.n_frm, best))


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    if args.head != "retrieval" or args.inference:
        print(json.dumps(dict(impl="reference", unavailable="the CPU arm times the retrieval train step (configs headline / c2 / c3) only")))
        return
    b = args.cpu_batch
    sd, batch = _cpu_setup(args, b)
    for _ in range(args.warmup):
        _cpu_step(sd, batch, args.n_clips, args.n_frm, args.size)
    steps = args.steps
    t0 = time.time()
    for _ in range(steps):
        _cpu_step(sd, batch, args.n_clips, args.n_frm, args.size)
    dt = (time.time() - t0) / steps
    val = round(b * args.n_clips / dt, 3)
    L = args.txt_len + (args.size // 32 // 2) ** 2
    out = dict(impl="reference", metric=METRIC_TRAIN, value=val, unit="clips/s", n_gpus=args.gpus,
               steps=steps, warmup=args.warmup, ms_per_step=round(dt * 1e3, 2), higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
               data="synthetic",
               config=dict(workload="MSRVTT retrieval train step (bounded CPU sample): %d videos x %d clips x %d frames %dx%d, %d-token text, n_ex=%d"
                           % (b, args.n_clips, args.n_frm, args.size, args.size, args.txt_len, args.n_ex), seq_len=L,
                           note="reference path = src/modeling/{modeling,transformers}.py + detectron2 R-50, restated in oracle/ (the Python "
                                "reference and detectron2 cannot travel to / install on the GPU box)"),
               cpu_baseline=dict(value=val, unit="clips/s", cores=torch.get_num_threads(), kind="port",
                                 sample="%d videos/step, %d timed steps, fp32 eager PyTorch, %d threads" % (b, steps, torch.get_num_threads())),
               e2e=dict(value=val, unit="clips/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 20; 3 with --impl reference, whose fp32 CPU steps take seconds)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps before them (default 5; 1 with --impl reference)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="headline", choices=sorted(CONFIGS), help="BASELINE.json workload (default: the configuration the metric names)")
    ap.add_argument("--batch", type=int, default=None, help="videos per GPU (default: the config's)")
    ap.add_argument("--n_clips", type=int, default=None)
    ap.add_argument("--n_frm", type=int, default=None)
    ap.add_argument("--size", type=int, default=224)
    ap.add_argument("--txt_len", type=int, default=None)
    ap.add_argument("--n_ex", type=int, default=None, help="text rows per video (captions / answer options)")
    ap.add_argument("--head", default=None, choices=["retrieval", "multiple_choice"])
    ap.add_argument("--inference", type=int, default=None, help="1: forward only (config c5)")
    ap.add_argument("--graph", type=int, default=1)
    ap.add_argument("--clip_batching", type=int, default=1, help="1: all clips of a step in one pass (forward_clips); 0: reference per-clip loop")
    ap.add_argument("--stem", default="s2d", choices=["s2d", "im2col"], help="stem conv: space-to-depth implicit GEMM or patch matrix + GEMM")
    ap.add_argument("--overlap_wgrad", type=int, default=1, help="wgrad GEMMs on a side stream beside the dgrad chain")
    ap.add_argument("--pdl", type=int, default=0, help="programmatic dependent launch between the library's kernels: 0 off, 1 all (hurts the wgrad overlap), 2 all but the GEMMs")
    ap.add_argument("--prefetch", type=int, default=1, help="e2e: upload batch i+1 on a copy stream while batch i computes (0: copy on the compute stream)")
    ap.add_argument("--attn_rows48", type=int, default=1, help="1 (default): attention of sequences up to 48 tokens on the 48-row / three-warp kernels; 0: 64-row kernels")
    ap.add_argument("--attn_flash_pipe", type=int, default=1, help="1 (default): long-sequence attention forward with cp.async double-buffered key tiles; 0: synchronous tile loads")
    ap.add_argument("--zero_grad_in_forward", type=int, default=1, help="1 (default): the step clears its two flat gradient buffers on a side stream beside "
                    "the transformer forward (ClipBert.zero_grad_in_forward); 0: a serial model.zero_grad() before every step")
    ap.add_argument("--fused_loss", type=int, default=1, help="1 (default): clip aggregation + LSE loss fwd+bwd as one kernel (cb_clip_lse_loss); 0: ~45 ATen launches")
    ap.add_argument("--recast_in_step", type=int, default=0, help="1: no optimizer attached before the loop -> fp32 -> bf16 weight re-cast inside every step (round-1 behaviour)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "nvls"], help="N>1 gradient exchange: NCCL all-reduce, this library's NVLS all-reduce (csrc/nvls.cu), or auto = nvls where a multicast mapping exists")
    ap.add_argument("--nvls_ctas", type=int, default=0, help="CTAs of the NVLS all-reduce kernel while it overlaps the backward; 0 (default) = by world size: 64 at N <= 4, "
                    "32 above (N = 8: 32 -> 0.966 of linear, 64 -> 0.953, 96 -> 0.942; N = 2: 64 -> 10.28 ms/step, 32 -> 11.2, 96 -> 10.37)")
    ap.add_argument("--nvls_tail_ctas", type=int, default=148, help="CTAs of the NVLS all-reduce of the last, exposed slices (0 = --nvls_ctas)")
    ap.add_argument("--wire", default="fp32", choices=["fp32", "bf16"], help="N>1: gradients travel as fp32 (the flat buffers as they are) or as bf16 (cast, all-reduce, cast back: half the payload, the reference's fp16 wire precision)")
    ap.add_argument("--cnn_buckets", type=int, default=1, help="N>1: exchange res5 + grid_encoder gradients mid-backward (default; 0: one CNN exchange at the end)")
    ap.add_argument("--sm_limit", type=int, default=0, help="cap the persistent GEMM grid (0 = all SMs); leaves SMs to the overlapped NCCL kernels")
    ap.add_argument("--nccl_ctas", type=int, default=0, help="N>1: NCCL_MAX_CTAS for the process group (0 = NCCL default)")
    ap.add_argument("--mn3d", type=int, default=1, help="dgrad / wgrad GEMMs: MN-major operands as one 3-D TMA box per k-chunk (default) or BN/64 2-D boxes")
    ap.add_argument("--group_wgrad", type=int, default=3, help="grouped weight-gradient launches (cb_gemm_wgrad_group): 0 none, 1 BertLayer + bottleneck block, 2 blocks only, 3 BertLayer only (default: measured best), 4 BertLayer as two pairs + blocks")
    ap.add_argument("--occ2", type=int, default=1, help="two GEMM CTAs per SM: 0 never, 1 only launches the tuning table marks, 2 every eligible launch up to --occ2_gflop")
    ap.add_argument("--occ2_gflop", type=float, default=0.0, help="with --occ2 2: largest launch (GFLOP) that runs two CTAs per SM (0 = no limit)")
    ap.add_argument("--cpu_batch", type=int, default=4)
    ap.add_argument("--optimizer", type=int, default=1, help="also time the fused AdamW step (informational key fused_optimizer)")
    ap.add_argument("--opt_steps", type=int, default=10, help="timed iterations of the informational fused-optimizer leg")
    ap.add_argument("--no_cpu", type=int, default=0, help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (logits, loss, sampled gradients) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 3 if args.impl == "reference" else 20
    if args.warmup is None:
        args.warmup = 1 if args.impl == "reference" else 5
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of this repository's timed path; --impl reference has none to write")
    args = apply_config(args)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
