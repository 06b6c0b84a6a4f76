#!/usr/bin/env python
"""bench_detector.py — whole-detector throughput: the second half of BASELINE.json's metric.

    python bench_detector.py --gpus 1 --steps K --warmup W                      # xLSTM-YOLO s-scale training, images/s
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench_detector.py --gpus N ...                                           # DDP, global batch 64 split over N ranks
    python bench_detector.py --mode infer --scale m --imgsz 1280 --batch 16      # BASELINE configs[4]
    python bench_detector.py --impl reference ...                                # the reference's own classes and PyTorch mLSTM

What runs: the reference's UNMODIFIED ``DetectionModel`` / ``parse_model`` / ``v8DetectionLoss`` (imported from
``baseline/_ref``, see baseline/make_ref.py) on the authored xLSTM-YOLO YAML of that scale, trained the way the reference's
trainer does a step (engine/trainer.py:363-389, :591-599): fp16 autocast forward + loss, loss x world_size, GradScaler backward,
unscale, clip_grad_norm(0.5), SGD step, EMA update; DDP with find_unused_parameters=True (:274).  Synthetic COCO-shaped batches
in the dict format of models/yolo/detect/train.py:57-74 (uint8 images from pinned host memory every step, ~7 boxes per image).

  --impl b200       this repo's ViLBlockPair (flip-free bidirectional pair, fused gates / tail, sm_100a mLSTM kernels)
                    constructed by the reference's own ViLBlockPairBlock
  --impl reference  the reference's ViL classes with HEAD's two breakages repaired (cell epilogue, pair composition; see
                    xlstm_yolo_b200/compat/reference_loader.py) and its own PyTorch chunkwise_simple as the cell arithmetic
                    (the Triton package HEAD names for CUDA is not installable here)

Prints ONE JSON line (rank 0): images/s over all ranks (global batch fixed: "scaling": "strong"), CUDA-event timed, max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def synthetic_batch(torch, b, imgsz, seed, boxes_per_img=7, pin=True):
    g = torch.Generator().manual_seed(seed)
    img = torch.randint(0, 256, (b, 3, imgsz, imgsz), dtype=torch.uint8, generator=g)
    if pin:
        img = img.pin_memory()
    n = b * boxes_per_img
    cls = torch.randint(0, 80, (n, 1), generator=g).float()
    xy = torch.rand(n, 2, generator=g) * 0.6 + 0.2
    wh = torch.rand(n, 2, generator=g) * 0.25 + 0.05
    return {"img": img, "cls": cls, "bboxes": torch.cat([xy, wh], 1), "batch_idx": torch.arange(b).repeat_interleave(boxes_per_img).float()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="train", choices=["train", "infer"])
    ap.add_argument("--scale", default="s", choices=["n", "s", "m", "l", "x"])
    ap.add_argument("--batch", type=int, default=64, help="GLOBAL batch (train: split over the ranks); per GPU for --mode infer")
    ap.add_argument("--imgsz", type=int, default=640)
    ap.add_argument("--device", default="cuda")
    ap.add_argument("--profile", default="", help="write a torch profiler table of one step to this file (rank 0)")
    ap.add_argument("--graph", type=int, default=0,
                    help="train mode: 1 = the network's forward and backward replayed from CUDA graphs (torch.cuda.make_graphed_callables "
                         "over the model's tensor path; loss, optimizer, EMA and DDP's all-reduce stay eager).  At 8 GPUs the eager step is "
                         "host-bound (60 ms of launches for 23 ms of device time at batch 8 per GPU)")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    import yaml

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    on_gpu = args.device == "cuda"
    if on_gpu and not torch.cuda.is_available():
        raise SystemExit("bench_detector.py needs a CUDA device (or --device cpu for a plumbing check)")
    dev = torch.device("cuda", local_rank) if on_gpu else torch.device("cpu")
    if on_gpu:
        torch.cuda.set_device(local_rank)
    out_fd = os.dup(1)          # stdout carries exactly one JSON line: library chatter (NCCL's banner, ...) goes to stderr
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl" if on_gpu else "gloo", **({"device_id": dev} if on_gpu else {}))

    from xlstm_yolo_b200.compat import reference_loader as RL
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "ultralytics")):
        if rank == 0:
            os.write(out_fd, (json.dumps({"impl": args.impl, "unavailable": "baseline/_ref/ultralytics missing: run baseline/make_ref.py where the reference tree exists"}) + "\n").encode())
        return 0
    V = RL.import_reference(ref_root)
    if args.impl == "b200":
        RL.use_b200_dropins(pair_level=True, head_compat=False)
    else:
        RL.apply_head_fixes(V, reference_backend=True, compose_pair=True)
    from ultralytics.cfg import get_cfg
    from ultralytics.nn.tasks import DetectionModel
    from ultralytics.utils.torch_utils import ModelEMA

    cfg = yaml.safe_load(open(os.path.join(ROOT, "xlstm_yolo_b200", "compat", "yamls", f"xlstm-yolo-{args.scale}.yaml")))
    cfg["scale"] = args.scale
    torch.manual_seed(0)
    model = DetectionModel(cfg, ch=3, nc=80, verbose=False)
    model.args = get_cfg()      # loss gains (box / cls / dfl) as the reference's defaults
    n_params = sum(p.numel() for p in model.parameters())
    model.to(dev)

    if args.mode == "train":
        assert args.batch % world == 0, "global batch must divide over the ranks"
        b = args.batch // world
        model.train()
        net = model
        graphed = None
        if args.graph and on_gpu:
            # The tensor path of the model (images -> the Detect head's three maps) as two CUDA graphs (forward, backward).  Every op of
            # this repo on that path is capturable (plain launches on the current stream, no host synchronisation, static shapes); the
            # loss (data-dependent target assignment) stays eager and takes the maps as its input (nn/tasks.py:  loss(batch, preds)).
            class TensorPath(torch.nn.Module):
                def __init__(self, m):
                    super().__init__()
                    self.m = m

                def forward(self, x):
                    with torch.autocast("cuda", cache_enabled=False):
                        return tuple(self.m.predict(x))
            model.criterion = model.init_criterion()
            sample = torch.rand(b, 3, args.imgsz, args.imgsz, device=dev)
            graphed = torch.cuda.make_graphed_callables(TensorPath(model), (sample,), num_warmup_iters=11 if world > 1 else 3,
                                                          allow_unused_input=True)   # the reference builds modules its forward never calls
            net = graphed
        if world > 1:   # engine/trainer.py:274
            net = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local_rank] if on_gpu else None, find_unused_parameters=True)
        # lr as in the first iterations of the reference's warm-up ramp (engine/trainer.py:366-375: from 0 towards lr0 = 0.01)
        opt = torch.optim.SGD(model.parameters(), lr=1e-4, momentum=0.937, nesterov=True, weight_decay=5e-4)
        scaler = torch.amp.GradScaler("cuda", enabled=on_gpu)
        ema = ModelEMA(model)
        batches = [synthetic_batch(torch, b, args.imgsz, 100 * rank + j, pin=on_gpu) for j in range(2)]

        def step(j):
            hb = batches[j % 2]
            batch = {k: v.to(dev, non_blocking=True) for k, v in hb.items()}
            batch["img"] = batch["img"].float() / 255          # models/yolo/detect/train.py:59
            if graphed is not None:
                preds = list(net(batch["img"]))
                with torch.autocast(dev.type, enabled=on_gpu):
                    loss, _ = model.criterion(preds, batch)
                    loss = loss.sum() * world
            else:
                with torch.autocast(dev.type, enabled=on_gpu):
                    loss, _ = net(batch)
                    loss = loss.sum() * world                   # engine/trainer.py:382-383
            scaler.scale(loss).backward()
            scaler.unscale_(opt)                                # engine/trainer.py:591-599
            torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=0.5)
            scaler.step(opt)
            scaler.update()
            opt.zero_grad()
            ema.update(model)
            return loss
        per_step_images = args.batch
        metric = "xLSTM-YOLO train images/s"
    else:
        b = args.batch
        model.eval()
        if on_gpu:
            model.half()                                         # engine/validator.py:117-119
        imgs = [torch.rand(b, 3, args.imgsz, args.imgsz, device=dev, dtype=torch.float16 if on_gpu else torch.float32) for _ in range(2)]

        def step(j):
            with torch.no_grad():
                y = model(imgs[j % 2])
            return y[0] if isinstance(y, (list, tuple)) else y
        per_step_images = b * world
        metric = "xLSTM-YOLO inference images/s"

    K, W = max(1, args.steps), max(1, args.warmup)
    for j in range(W):
        last = step(j)
    if on_gpu:
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if on_gpu:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
    t0 = time.perf_counter()
    for j in range(K):
        last = step(W + j)
    if on_gpu:
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
    else:
        ms = (time.perf_counter() - t0) * 1e3
    if world > 1:
        dist.barrier()
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    finite = bool(torch.isfinite(last.float()).all())

    if args.profile and rank == 0 and on_gpu:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            step(0)
            torch.cuda.synchronize()
        with open(args.profile, "w") as fh:
            fh.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40))

    if rank == 0:
        ms_per_step = ms / K
        out = {
            "metric": metric, "value": per_step_images / (ms_per_step * 1e-3), "unit": "images/s", "impl": args.impl,
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong" if args.mode == "train" else "weak", "vs_baseline": None,
            "dtype": "fp16 autocast (mLSTM kernels: bf16 operands, fp32 accumulation)" if on_gpu else "fp32", "data": "synthetic",
            "config": {"model": f"xlstm-yolo-{args.scale}", "params": n_params, "imgsz": args.imgsz, "cuda_graph": int(bool(args.graph)),
                       "global_batch": args.batch if args.mode == "train" else b * world, "batch_per_gpu": b,
                       "parallelism": f"ddp{world}" if args.mode == "train" else f"replicas{world}", "mode": args.mode,
                       "vil": ("this repo's ViLBlockPair drop-in (BR(TL(x)), flip-free)" if args.impl == "b200" else
                               "reference ViL classes + HEAD fixes + reference PyTorch chunkwise_simple")},
            "loss_finite": finite,
        }
        os.write(out_fd, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
