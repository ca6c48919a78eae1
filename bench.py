#!/usr/bin/env python
"""bench.py — the hot path's headline metric on B200 (see BASELINE.json, SURVEY.md §8d, DESIGN.md §6).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg1]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the per-pixel multi-dataset label-space path over one synthetic batch:
    raw uint8 label maps --lb_map LUT--> labels
    unified logits --bipartite projection + bilinear upsample + OhemCE fwd + selection + bwd--> loss, dlogits
    (labels, preds) --confusion matrix (+ all-reduce) --> mIoU per dataset
Metric: labelled pixels / second, whole job (all ranks).  Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

import numpy as np
import torch
import torch.distributed as dist

METRIC = "labelled pixels/sec (head+OHEM fwd+bwd, mIoU hist)"
UNIT = "pixels/s"

WORKLOADS = {
    # name: (n_cats, C_uni, dataset ids of the per-GPU batch, (h, w), (H, W))
    "cfg3": ([19, 64, 37, 19, 26, 150, 133], 358, [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6], (256, 512), (1024, 2048)),
    "cfg2": ([19, 12, 36], 67, [0] * 5 + [1] * 5 + [2] * 6, (256, 512), (1024, 2048)),
    "cfg1": ([19], 19, [0, 0], (128, 256), (512, 1024)),
    # the repo's own per-GPU batch of that config: crop 768 x 768, ims_per_gpu 4 for each of the 7 datasets
    "cfg3_native": ([19, 64, 37, 19, 26, 150, 133], 358, [d for d in range(7) for _ in range(4)], (192, 192), (768, 768)),
    "tiny": ([5, 3, 7], 11, [0, 1, 2, 2], (16, 32), (64, 128)),
}
WORKLOAD_NAMES = {
    "cfg3": "ltbgnn_7_datasets_snp: 7-dataset unified label space (C_uni 358), per-GPU batch 16x1024x2048, logits 256x512",
    "cfg2": "ltbgnn_city_cam_a2d2: 3 datasets (C_uni 67), per-GPU batch 16x1024x2048, logits 256x512",
    "cfg1": "bisenetv2_city-sized: 1 dataset 19 classes, batch 2x512x1024, logits 128x256",
    "cfg3_native": "ltbgnn_7_datasets_snp at the repo's own crop: 7 datasets x 4 images of 768x768, logits 192x192",
    "tiny": "tiny self-test",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=list(WORKLOADS))
    ap.add_argument("--label-dtype", default="int64", choices=["int64", "uint8"],
                    help="dtype of the remapped label maps (the reference's loaders hand int64 to the loss)")
    ap.add_argument("--with-aux", action="store_true",
                    help="add the per-dataset aux heads (OhemCELoss 0.7 on aux_logits[i], weight 0.2; "
                         "loss_cross_datasets.py:1044-1056,1129-1130) to the step; not part of the headline config")
    ap.add_argument("--logits-dtype", default="f32", choices=["f32", "bf16", "f16"],
                    help="dtype of logits_uni / dlogits_uni (AMP trainers hand fp16 logits to the loss; the CE "
                         "arithmetic stays fp32 either way).  The headline is f32.")
    ap.add_argument("--eager-gpu", action="store_true",
                    help="also time the reference's own torch op sequence (oracle/torch_ref.py, the same code as the "
                         "CPU baseline) on CUDA tensors on this GPU: PyTorch eager, reported as 'reference_eager_gpu'")
    ap.add_argument("--bi-graphs", default="onehot", choices=["onehot", "dense"],
                    help="onehot: 0/1 column-one-hot graphs (SEG stage, the headline).  dense: soft trainable graphs "
                         "softmax(randn * 4) with requires_grad (GNN stage): projection, adjoint and d bi_graph run on "
                         "the tcgen05 tensor cores; not the headline config")
    ap.add_argument("--logits", default="randn", choices=["randn", "confident", "mixed"],
                    help="randn: SURVEY 8d's headline batch (every loss far above the threshold: threshold branch of the "
                         "OHEM selection).  confident: labels constant in blocks of 128 x 128 px and +12 on the unified "
                         "channels of the block's class, so fewer than n_min pixels are hard and the top-k fallback "
                         "(radix select over all 33.5 M losses, ohem_ce_loss.py:87-88) runs and is timed.  mixed: as "
                         "confident with blocks of 256 x 256 px, but the logits of every eighth block predict a wrong "
                         "class: ~12 % of the pixels (+ the block borders) "
                         "are hard (threshold branch) and whole regions carry no gradient, what a partly trained net "
                         "looks like (the backward skips warps without a selected pixel)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the workload's batch per GPU.  strong: the batch is split over the ranks "
                         "(SURVEY 8e: global batch 16 -> 2 images per GPU at N = 8)")
    ap.add_argument("--shard", default="balanced", choices=["balanced", "contiguous"],
                    help="--scaling strong: how the batch is split over the ranks.  balanced: equal image counts, images "
                         "dealt by falling class count to the least loaded rank (dist_utils.shard_images_balanced); "
                         "contiguous: blocks of consecutive images (both 150-class images of the cfg3 batch on one rank)")
    ap.add_argument("--pred-dtype", default="int64", choices=["int64", "int32", "uint8"],
                    help="dtype of the predictions handed to the confusion matrix (the reference's argmax gives int64)")
    ap.add_argument("--cuda-graph", action="store_true",
                    help="capture one whole step (LUT, loss forward, selection, backward through autograd, confusion "
                         "matrices on the side stream, all-reduce, mIoU) into a CUDA graph and replay it in the "
                         "device-resident timed loop: for the launch-bound regimes (strong scaling to a few images per "
                         "GPU, cfg1), where ~25 launches per step cost more host time than the kernels take")
    ap.add_argument("--no-aux-workload", action="store_true",
                    help="skip the second named workload (the same step with the per-dataset aux heads)")
    ap.add_argument("--no-numa-bind", action="store_true",
                    help="do not pin the rank to the CPUs of its GPU's NUMA node (A/B of the e2e arm)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-times", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0): "
                         "loss, miou, confusion (the flat int64 histograms of every dataset, as float64) and the "
                         "gradients d logits_uni, d bi_graph<i> (--bi-graphs dense) and d aux<i> (--with-aux) as "
                         "float32.  A gradient of more than %d elements is stored at a fixed, seeded sample of "
                         "positions, so two builds run with the same arguments can be compared output for output"
                         % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


# ---------------------------------------------------------------------------------------------
# synthetic batch (SURVEY.md §8d): identical recipe for the GPU arm and the CPU arms
# ---------------------------------------------------------------------------------------------
def make_graphs(n_cats, c_uni, gen):
    graphs = []
    for c in n_cats:
        idx = torch.randint(0, c, (c_uni,), generator=gen)
        idx[:c] = torch.arange(c)  # every dataset class non-empty (column-one-hot 0/1 graph, SEG stage)
        m = torch.zeros(c, c_uni)
        m[idx, torch.arange(c_uni)] = 1
        graphs.append(m)
    return graphs


def make_luts(n_cats):
    luts = []
    for c in n_cats:
        lut = np.full(256, 255, dtype=np.uint8)
        lut[:243] = np.arange(243) % c  # raw ids 243..255 are void (~5 % ignore)
        luts.append(lut)
    return luts


def make_batch(workload, device, seed, images=None, logits="randn"):
    n_cats, c_uni, ids, (h, w), (H, W) = WORKLOADS[workload]
    if images is not None:
        ids = [ids[i] for i in images]
    gen = torch.Generator().manual_seed(1234)
    graphs = make_graphs(n_cats, c_uni, gen)
    luts = make_luts(n_cats)
    dgen = torch.Generator(device=device).manual_seed(seed)
    B = len(ids)
    x = torch.randn(B, c_uni, h, w, generator=dgen, device=device)
    raw = torch.randint(0, 256, (B, H, W), generator=dgen, device=device, dtype=torch.uint8)
    pred = torch.empty(B, H, W, dtype=torch.int64, device=device)
    for b, d in enumerate(ids):
        pred[b] = torch.randint(0, n_cats[d], (H, W), generator=dgen, device=device)
    if logits in ("confident", "mixed"):
        # spatially coherent labels (blocks of 32 x 32 low-res cells) that the logits predict: raw id r -> class r % C
        blk = 64 if logits == "mixed" else 32  # mixed: 256 x 256 px regions, two warp strips of the kernels wide
        for b, d in enumerate(ids):
            c = n_cats[d]
            cls = torch.randint(0, c, ((h + blk - 1) // blk, (w + blk - 1) // blk), generator=dgen, device=device)
            low = cls.repeat_interleave(blk, 0)[:h].repeat_interleave(blk, 1)[:, :w]              # [h, w] class map
            fy, fx = H // h, W // w
            raw[b] = low.repeat_interleave(fy, 0).repeat_interleave(fx, 1)[:H, :W].to(torch.uint8)  # raw id == class
            col_cls = graphs[d].argmax(0).to(device)                                              # class of unified u
            guess = low
            if logits == "mixed":  # every eighth block is predicted wrongly
                wrong = (torch.rand(cls.shape, generator=dgen, device=device) < 0.125)
                wrong = wrong.repeat_interleave(blk, 0)[:h].repeat_interleave(blk, 1)[:, :w]
                guess = torch.where(wrong, (low + 1) % c, low)
            x[b] += 12.0 * (col_cls[:, None, None] == guess[None]).to(x.dtype)
            raw[b][torch.rand(H, W, generator=dgen, device=device) < 0.03] = 250                  # void -> 255
    return dict(n_cats=n_cats, c_uni=c_uni, ids=ids, h=h, w=w, H=H, W=W, x=x, raw=raw, pred=pred, graphs=graphs,
                luts=luts)


DUMP_MAX_ELEMS = 1 << 20  # 4 MB of float32 per array: d logits_uni plus seven aux heads stay far below 64 MB


def dump_outputs(out_dir, arrays):
    """np.save every array as out_dir/<name>.npy; integers as float64, the rest as float32.  An array of more than
    DUMP_MAX_ELEMS elements is reduced to the elements at DUMP_MAX_ELEMS flat positions drawn with a seed that depends
    only on its size, so the same arguments select the same positions in every run."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t is None:  # a tensor that received no gradient
            continue
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            pos = np.random.default_rng(t.numel()).choice(t.numel(), DUMP_MAX_ELEMS, replace=False)
            pos.sort()
            t = t.reshape(-1)[torch.from_numpy(pos).to(t.device)]
        t = t.to(torch.float32 if t.is_floating_point() else torch.float64)
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


def dataset_slices(ids):
    """contiguous image ranges per dataset (ids are sorted in the trainer's batch layout)."""
    out, start = [], 0
    for i in range(1, len(ids) + 1):
        if i == len(ids) or ids[i] != ids[start]:
            out.append((ids[start], start, i))
            start = i
    return out


# ---------------------------------------------------------------------------------------------
# clocks sampler
# ---------------------------------------------------------------------------------------------
class Clocks(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples = index, False, []

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def config_of(args, world):
    """The `config` object of the JSON line — the same keys and values for the GPU arm and the reference arm."""
    n_cats, c_uni, ids, (h, w), (H, W) = WORKLOADS[args.workload]
    n_img = len(ids) if args.scaling == "weak" else len(ids) // max(world, 1)
    px = n_img * H * W
    e = 4 if args.logits_dtype == "f32" else 2
    L = 8 if args.label_dtype == "int64" else 1
    P = {"int64": 8, "int32": 4, "uint8": 1}[args.pred_dtype]
    return {
        "workload": WORKLOAD_NAMES[args.workload], "name": args.workload, "pixels_per_step_per_gpu": px,
        "labels": args.label_dtype, "preds": args.pred_dtype,
        "logits": f"{args.logits_dtype} NCHW (CE arithmetic fp32)",
        "logit_values": {"randn": "randn (every loss above the OHEM threshold: threshold branch)",
                         "confident": "confident (block labels predicted by the logits: top-k fallback branch)",
                         "mixed": "mixed (block labels, every eighth block predicted wrongly: threshold branch, ~12 % "
                                  "of the pixels selected)"}[args.logits],
        "bi_graphs": "0/1 column-one-hot (SEG stage)" if args.bi_graphs == "onehot" else
                     "dense fp32 softmax graphs with grad (GNN stage; tcgen05 projection, adjoint, d bi_graph)",
        "ohem_thresh": 0.4, "aux_heads": bool(args.with_aux),
        "l2": "inputs_exceed_l2 (logits %.2f GB, labels+preds %.2f GB per step)" %
              (n_img * c_uni * h * w * e / 1e9, px * (1 + L + P) / 1e9),
        "parallelism": f"dp{world} (images sharded, OHEM selection rank-local, one int64 hist all-reduce)",
        "scaling": args.scaling if args.scaling == "weak" else f"strong ({args.shard} split of the batch)",
        "cuda_graph": bool(args.cuda_graph),
        "streams": "loss fwd/select/bwd on the main stream, confusion matrices + all-reduce + mIoU on a side stream; "
                   "e2e: host->device copies of step i+1 on a copy stream beside step i",
    }


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
KERNELS_PER_CALL = {"mdseg_proj_fwd_tc16": 1, "mdseg_proj_bwd_tc16": 1, "mdseg_proj_bwd_graph_tc16": 2, "mdseg_head_fwd_tc16": 1, "mdseg_head_dw_tc16": 2, "mdseg_up_nll_fwd": 1,
                    "mdseg_up_nll_bwd": 1, "mdseg_softmax_nchw": 1, "mdseg_softmax_bwd_nchw": 1,
                    "mdseg_up_ce_bwd_direct": 3, "mdseg_proj_fwd_tc": 2, "mdseg_proj_bwd_tc": 3, "mdseg_proj_bwd_graph_tc": 2,
                    "mdseg_lut_remap_images": 1, "mdseg_confusion_images": 1, "mdseg_miou_images": 1,
                    "mdseg_lut_remap": 1, "mdseg_confusion": 1, "mdseg_miou": 1, "mdseg_ohem_begin": 1,
                    "mdseg_proj_fwd": 1, "mdseg_up_ce_fwd": 1, "mdseg_ohem_select": 1, "mdseg_up_ce_bwd": 1,
                    "mdseg_proj_bwd": 1, "mdseg_mds_bwd": 4, "mdseg_ohem_ce_fwd": 1, "mdseg_ohem_ce_bwd": 1, "mdseg_add_planes": 1}


_AFFINITY_BEFORE = []


def bind_to_gpu_numa_node(local_rank):
    """Run this rank on the CPUs of its GPU's NUMA node, so that its pinned host buffers (first touch) and its copy
    engine's reads stay on the socket the GPU hangs off: with eight ranks on one host the H2D copies of the e2e arm
    otherwise all read one node's DRAM.  Best effort: returns what was done for the JSON line."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(base + "/numa_node").read())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0)
        _AFFINITY_BEFORE.append(allowed)  # restored before the CPU baseline, which uses every host core
        use = cpus & allowed
        if node < 0 or not use:
            return {"node": node, "bound": False, "why": "no NUMA node reported or no local CPU allowed"}
        os.sched_setaffinity(0, use)
        return {"node": node, "bound": True, "cpus": len(use), "pci": bdf}
    except Exception as e:  # sysfs layout, permissions, torch without the pci_* properties
        return {"bound": False, "why": repr(e)[:120]}


def run_ours(args, rank, world, local_rank):
    from mdseg_b200 import dist_utils, native, ops  # raises if libmdseg_b200.so is missing: no fallback

    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    numa = bind_to_gpu_numa_node(local_rank) if not args.no_numa_bind else {"bound": False, "why": "--no-numa-bind"}
    launches = {"n": 0}
    per_call_ms = {}
    timing = {"on": False}
    raw_call = native.call

    def counting_call(name, *a):
        launches["n"] += KERNELS_PER_CALL.get(name, 1)
        if timing["on"]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            raw_call(name, *a)
            e1.record()
            per_call_ms.setdefault(name, []).append((e0, e1))
        else:
            raw_call(name, *a)

    native.call = counting_call
    ops.N.call = counting_call

    images = None
    if args.scaling == "strong":  # the workload's batch split over the ranks (contiguous image ranges)
        n_all = len(WORKLOADS[args.workload][2])
        if n_all % world:
            raise SystemExit(f"--scaling strong: {n_all} images do not split over {world} ranks")
        if args.shard == "balanced":
            wl = WORKLOADS[args.workload]
            images = dist_utils.shard_images_balanced([wl[0][d] for d in wl[2]], rank, world)
        else:
            images = list(dist_utils.shard_images(n_all, rank, world))
    bt = make_batch(args.workload, dev, 1234 + rank, images=images, logits=args.logits)
    bt["pred"] = bt["pred"].to({"int64": torch.int64, "int32": torch.int32, "uint8": torch.uint8}[args.pred_dtype])
    n_cats, ids, H, W = bt["n_cats"], bt["ids"], bt["H"], bt["W"]
    B = len(ids)
    px = B * H * W
    lab_dt = torch.int64 if args.label_dtype == "int64" else torch.uint8
    graphs = [g.to(dev) for g in bt["graphs"]]
    if args.bi_graphs == "dense":  # GNN stage: soft adjacency with grad (loss_cross_datasets.py:997-1006)
        ggen = torch.Generator(device=dev).manual_seed(7)
        graphs = [torch.softmax(torch.randn(c, bt["c_uni"], generator=ggen, device=dev) * 4, dim=0).requires_grad_(True)
                  for c in n_cats]
    luts = torch.from_numpy(np.stack(bt["luts"])).to(dev)  # [n_datasets, 256]
    ids_t = torch.tensor(ids, dtype=torch.int32, device=dev)
    slices = dataset_slices(ids)
    thresh = ops.neg_log(0.4)
    aux = None
    if args.with_aux:
        agen = torch.Generator(device=dev).manual_seed(99 + rank)
        aux = [torch.randn(B, c, bt["h"], bt["w"], generator=agen, device=dev).requires_grad_(True) for c in n_cats]
    ldt = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[args.logits_dtype]
    bt["x"] = bt["x"].to(ldt)
    x = bt["x"].requires_grad_(True)
    offs = np.cumsum([0] + [c * c for c in n_cats])
    hist_flat = torch.zeros(int(offs[-1]), dtype=torch.int64, device=dev)
    hists = [hist_flat[offs[d]:offs[d + 1]].view(n_cats[d], n_cats[d]) for d in range(len(n_cats))]
    out = {}

    side = torch.cuda.Stream(device=dev)  # label-space evaluation runs beside the loss (independent given the labels)

    def evaluate(labels, pred, reduce):
        # a12/a13: confusion matrices of every dataset (one launch) + one int64 all-reduce + mIoU
        hist_flat.zero_()
        ops.confusion_images(labels, pred, ids_t, n_cats, hist=hist_flat)
        if reduce:  # evaluate.py:187-188
            dist_utils.allreduce_hist(hist_flat)
        return ops.miou_images(hist_flat, n_cats)[1]

    def step(raw, xin, pred, reduce=True, overlap=True, aux=aux):
        # a1: dataset lb_map LUT (lib/base_dataset.py:81-82), one table per dataset, one launch for the batch
        labels = ops.lut_remap_images(raw, luts, ids_t, out_dtype=lab_dt)
        main = torch.cuda.current_stream()
        # a5-a9: fused projection + upsample + OhemCE fwd, selection, bwd
        xin.grad = None
        for gph in graphs:
            gph.grad = None
        loss = ops.mds_proj_ohem_ce(xin, labels, ids_t, graphs, thresh)
        out["states"] = loss.grad_fn.states
        if aux is not None:
            for t in aux:
                t.grad = None
            per_ds = ops.up_ohem_ce(aux, labels, ids_t, ops.neg_log(0.7), seg_per_dataset=True)
            loss = loss + 0.2 * torch.nan_to_num(per_ds, nan=0.0).sum()
        if overlap:  # the HBM/atomic-bound evaluation runs beside the issue-bound backward
            side.wait_stream(main)
            with torch.cuda.stream(side):
                mious = evaluate(labels, pred, reduce)
        loss.backward()
        if overlap:
            main.wait_stream(side)
            labels.record_stream(side)
            mious.record_stream(main)
        else:
            mious = evaluate(labels, pred, reduce)
        out["loss"], out["miou"] = loss.detach(), mious

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: `value` ---------------------------------------------------------
    for _ in range(max(args.warmup, 3)):
        step(bt["raw"], x, bt["pred"])
    barrier()
    ops.check_errors(dev)
    launches["n"] = 0
    clocks = Clocks(local_rank) if rank == 0 else None
    if clocks:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    graph = None
    if args.cuda_graph:
        # every buffer of the step is static (inputs) or comes from the graph's private pool (autograd included); the
        # library never synchronises or allocates, so the capture holds exactly the launches of one step
        graph = torch.cuda.CUDAGraph()
        cap = torch.cuda.Stream(device=dev)
        cap.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cap):
            launches["n"] = 0
            with torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                step(bt["raw"], x, bt["pred"])
            per_step_launches = launches["n"]
        torch.cuda.current_stream().wait_stream(cap)
        for _ in range(3):
            graph.replay()
        barrier()
        ops.check_errors(dev)
    barrier()
    e0.record()
    if graph is not None:
        for _ in range(args.steps):
            graph.replay()
        launches["n"] = per_step_launches * args.steps
    else:
        for _ in range(args.steps):
            step(bt["raw"], x, bt["pred"])
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:  # before the checks and the other loops below overwrite the step's results
        outputs = {"loss": out["loss"], "miou": out["miou"], "confusion": hist_flat, "dlogits_uni": x.grad}
        if args.bi_graphs == "dense":
            outputs.update({f"dbi_graph{d}": g.grad for d, g in enumerate(graphs)})
        if aux is not None:
            outputs.update({f"daux{d}": t.grad for d, t in enumerate(aux)})
        dump_outputs(args.dump_outputs, outputs)
    ms = e0.elapsed_time(e1)
    gpu_launches = launches["n"]
    ms = dist_utils.max_over_ranks(ms, dev)
    ms_per_step = ms / args.steps
    value = dist_utils.whole_job_rate(px, world, ms_per_step)
    loss_val = float(out["loss"])
    st0 = ops.read_states(out["states"])[0]
    sel_mode = int(st0.mode)
    ohem = {"branch": "top-k fallback" if sel_mode else "threshold", "n_valid": int(st0.n_valid), "n_hard": int(st0.n_hard),
            "n_min": int(st0.n_min), "n_sel": int(st0.n_sel)}

    # ---- correctness of what the all-reduce returned (outside the timed region): every labelled pixel of every rank
    # is in exactly one cell of the reduced histograms
    labels_chk = ops.lut_remap_images(bt["raw"], luts, ids_t, out_dtype=torch.uint8)
    n_valid_local = (labels_chk != 255).sum().to(torch.int64).reshape(1)
    gathered = [torch.zeros_like(n_valid_local) for _ in range(world)]
    if world > 1:
        dist.all_gather(gathered, n_valid_local)
    else:
        gathered = [n_valid_local]
    evaluate(labels_chk, bt["pred"], True)
    torch.cuda.synchronize()
    hist_sum, want_sum = int(hist_flat.sum()), int(sum(int(g) for g in gathered))
    hist_check = {"hist_sum": hist_sum, "sum_of_rank_n_valid": want_sum, "ok": hist_sum == want_sum,
                  "n_valid_per_rank": [int(g) for g in gathered]}
    if not hist_check["ok"]:
        raise SystemExit(f"reduced histogram holds {hist_sum} pixels, the ranks labelled {want_sum}")
    del labels_chk

    # ---- second named workload: the same step WITH the per-dataset aux heads (with_datasets_aux of the config;
    # SURVEY 8d cfg3 lists them; the reference net emits every head for all images, semseg.py:326-333)
    aux_workload = None
    if aux is None and not args.no_aux_workload and args.bi_graphs == "onehot":
        x.grad = None
        torch.cuda.empty_cache()  # the allocator starts from the state a run of this workload alone would have: behind
        # the main workload's cached blocks the mean of this loop was seen at 5.7, 7.7 and 20 ms in three runs while
        # `--with-aux` alone gave 5.70 three times (allocator misses inside single steps suspected); the per-step median
        # and maximum are reported next to the mean so that a stalled step shows
        agen = torch.Generator(device=dev).manual_seed(99 + rank)
        aux2 = [torch.randn(B, c, bt["h"], bt["w"], generator=agen, device=dev, dtype=ldt).requires_grad_(True)
                for c in n_cats]
        for _ in range(5):
            step(bt["raw"], x, bt["pred"], aux=aux2)
        barrier()
        n_aux = max(3, min(args.steps, 10))
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n_aux + 1)]
        evs[0].record()
        for i in range(n_aux):
            step(bt["raw"], x, bt["pred"], aux=aux2)
            evs[i + 1].record()
        barrier()
        per_step = [evs[i].elapsed_time(evs[i + 1]) for i in range(n_aux)]
        ms_aux = dist_utils.max_over_ranks(evs[0].elapsed_time(evs[n_aux]), dev) / n_aux
        e_sz = 4 if ldt == torch.float32 else 2
        Lb = 8 if lab_dt == torch.int64 else 1
        cbar_all = sum(n_cats)  # every head is [B, C_d, h, w] over all images; rows of other datasets are only zero-filled
        bytes_aux = 3 * sum(n_cats[d] for d in ids) / len(ids) * e_sz / 16 + Lb + 20
        bytesA = 3 * bt["c_uni"] * e_sz / 16 + 2 * Lb + 20
        aux_workload = {"name": args.workload + "_with_aux", "ms_per_step": ms_aux, "steps": n_aux,
                        "ms_per_step_median": float(np.median(per_step)), "ms_per_step_max": float(max(per_step)),
                        "value": dist_utils.whole_job_rate(px, world, ms_aux), "unit": UNIT, "loss": float(out["loss"]),
                        "alg_bytes_per_px_group_A_plus_aux": round(bytesA + bytes_aux, 2),
                        "aux_logit_bytes": int(B * cbar_all * bt["h"] * bt["w"] * e_sz)}
        del aux2
        x.grad = None
        torch.cuda.empty_cache()

    # ---- end-to-end through the public API with HOST buffers: `e2e` ------------------------------------
    h_x = bt["x"].detach().cpu().pin_memory()
    h_raw = bt["raw"].cpu().pin_memory()
    h_pred = bt["pred"].cpu().pin_memory()
    # two device input sets: the host->device copies of step i + 1 run on a copy stream beside the kernels of step i
    # (what a data loader with a prefetch queue does); every timed step still copies its own inputs and reads its
    # own results back, and the timed region contains exactly e2e_steps copies and e2e_steps computations.
    bufs = []
    for _ in range(2):
        bufs.append((torch.empty_like(bt["x"].detach()).requires_grad_(True), torch.empty_like(bt["raw"]),
                     torch.empty_like(bt["pred"]), torch.cuda.Event()))
    h2d = h_x.numel() * h_x.element_size() + h_raw.numel() + h_pred.numel() * h_pred.element_size()
    d2h = 4 + 4 * len(n_cats)
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream()

    def issue_copy(slot):
        d_x, d_raw, d_pred, ready = bufs[slot]
        copy_stream.wait_stream(main_stream)  # the buffers' previous consumer (two steps ago) has been enqueued
        with torch.cuda.stream(copy_stream), torch.no_grad():
            d_x.copy_(h_x, non_blocking=True)
            d_raw.copy_(h_raw, non_blocking=True)
            d_pred.copy_(h_pred, non_blocking=True)
            ready.record(copy_stream)

    def e2e_step(i, prefetch_next):
        d_x, d_raw, d_pred, ready = bufs[i % 2]
        main_stream.wait_event(ready)
        if prefetch_next:
            issue_copy((i + 1) % 2)
        step(d_raw, d_x, d_pred)
        return float(out["loss"].cpu()), out["miou"].cpu()

    e2e_steps = max(2, min(args.steps, 5))
    issue_copy(0)
    e2e_step(0, False)  # warm-up
    barrier()
    e0.record()
    issue_copy(1)  # pipeline fill: the first timed step waits for its own copy
    for i in range(1, e2e_steps + 1):
        e2e_step(i, i < e2e_steps)
    e1.record()
    barrier()
    e2e_ms = dist_utils.max_over_ranks(e0.elapsed_time(e1), dev) / e2e_steps
    e2e_value = dist_utils.whole_job_rate(px, world, e2e_ms)
    clk = clocks.summary() if clocks else None  # sampled over the device-resident and the end-to-end timed loops
    del h_x, bufs

    # ---- per-kernel durations (separate loop, L2 flushed between launches) -> roofline -------------------
    peak, peak_src = measured_peak()
    roof, per_kernel = None, {}
    if rank == 0 and not args.no_kernel_times:
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

        def flushing_call(name, *a):
            flush.fill_(1)
            counting_call(name, *a)

        native.call = flushing_call
        ops.N.call = flushing_call
        timing["on"] = True
        for _ in range(5):
            step(bt["raw"], x, bt["pred"], reduce=False, overlap=False)  # rank 0 only: no collective in this loop
        torch.cuda.synchronize()
        timing["on"] = False
        native.call = counting_call
        ops.N.call = counting_call
        del flush
        e = 4 if bt["x"].dtype == torch.float32 else 2
        L = 8 if lab_dt == torch.int64 else 1
        cbar = sum(n_cats[d] for d in ids) / len(ids)  # mean C_ds over the images of the batch
        cu = bt["c_uni"]
        # algorithmic bytes per LABEL pixel of each C-ABI call (DESIGN.md §5); 16 label px per logit px
        alg = {
            "mdseg_proj_fwd": (cu * e + cbar * 4) / 16,
            "mdseg_up_ce_fwd": cbar * 4 / 16 + L + 8,
            "mdseg_ohem_select": 4,
            "mdseg_up_ce_bwd": cbar * 4 / 16 + L + 8 + 2 * cbar * 4 / 16,
            "mdseg_proj_bwd": (2 * cbar * 4 + cu * e) / 16,
            "mdseg_mds_bwd": cbar * 4 / 16 + L + 8 + cu * e / 16,
            "mdseg_proj_fwd_tc": (cu * e + cbar * 4) / 16,
            "mdseg_up_ce_bwd_direct": cbar * 4 / 16 + L + 8 + cbar * 4 / 16,
            "mdseg_proj_bwd_tc": (cbar * 4 + cu * e) / 16,
            "mdseg_proj_bwd_graph_tc": (cbar * 4 + cu * e) / 16,
            "mdseg_proj_fwd_tc16": (cu * e + cbar * 4) / 16,
            "mdseg_proj_bwd_tc16": (cbar * e + cu * e) / 16,
            "mdseg_proj_bwd_graph_tc16": (cbar * e + cu * e) / 16,
            "mdseg_lut_remap": 1 + L,
            "mdseg_confusion": L + 8,
            "mdseg_lut_remap_images": 1 + L,
            "mdseg_confusion_images": L + 8,
        }
        if sel_mode == 0:
            alg.pop("mdseg_ohem_select")  # threshold branch: the select kernel exits after the decision, no loss is read
        if args.with_aux:  # the aux heads run through the same two calls: their bytes belong to them
            aux_px = cbar * e / 16
            alg["mdseg_up_ce_fwd"] += aux_px + L + 8
            alg["mdseg_up_ce_bwd_direct"] = alg.get("mdseg_up_ce_bwd_direct", 0)
        for name, evs in per_call_ms.items():
            calls_per_step = len(evs) / 5
            tot = sum(a.elapsed_time(b) for a, b in evs) / 5  # ms per step spent in this ABI call
            per_kernel[name] = {"ms_per_step": round(tot, 4), "launches_per_step": calls_per_step}
            if name == "mdseg_ohem_select":
                per_kernel[name]["branch"] = ohem["branch"]
            if name in alg:
                gbs = alg[name] * px / (tot * 1e-3) / 1e9
                per_kernel[name].update({"alg_bytes_per_px": round(alg[name], 3), "achieved_gbs": round(gbs, 1),
                                         "frac": round(gbs / peak, 4)})
        # the three tensor-core calls of the GNN stage: useful FLOP = 2 * C_uni * C_ds per low-res pixel each
        tf_peak = None
        if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")):
            tf_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops_sustained")
        for name in ("mdseg_proj_fwd_tc", "mdseg_proj_bwd_tc", "mdseg_proj_bwd_graph_tc", "mdseg_proj_fwd_tc16",
                     "mdseg_proj_bwd_tc16", "mdseg_proj_bwd_graph_tc16"):
            if name in per_kernel:
                tfl = 2.0 * cu * cbar * (px / 16) / (per_kernel[name]["ms_per_step"] * 1e-3) / 1e12
                per_kernel[name]["useful_tflops"] = round(tfl, 1)
                if tf_peak:
                    per_kernel[name]["frac_of_bf16_peak"] = round(tfl / tf_peak, 4)
        cand = {k: v for k, v in per_kernel.items() if "achieved_gbs" in v}
        if cand:
            top = max(cand, key=lambda k: cand[k]["ms_per_step"])
            traffic = None
            prof = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(prof):
                traffic = json.load(open(prof)).get(top)  # ncu dram bytes of the call's dominant kernel
            roof = {"kernel": top, "bound": "hbm", "achieved": cand[top]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": cand[top]["frac"], "traffic": traffic, "peak_source": peak_src,
                    "duration_ms": cand[top]["ms_per_step"]}
        # whole group A (SURVEY §8d: 3*C_uni*e/16 + 2L + 20 bytes per pixel) and B (L + 8)
        grpA = sum(per_kernel.get(k, {}).get("ms_per_step", 0) for k in
                   ("mdseg_proj_fwd", "mdseg_up_ce_fwd", "mdseg_ohem_begin", "mdseg_ohem_select", "mdseg_up_ce_bwd",
                    "mdseg_proj_bwd", "mdseg_mds_bwd", "mdseg_proj_fwd_tc", "mdseg_up_ce_bwd_direct",
                    "mdseg_proj_bwd_tc", "mdseg_proj_bwd_graph_tc", "mdseg_proj_fwd_tc16", "mdseg_proj_bwd_tc16",
                    "mdseg_proj_bwd_graph_tc16"))
        bytesA = 3 * cu * e / 16 + 2 * L + 20
        if args.with_aux:  # + one pass over each image's own head forward, two backward (read + write), labels, loss
            bytesA += 3 * cbar * e / 16 + L + 20
        if grpA:
            per_kernel["group_A_loss_fwd_select_bwd"] = {
                "ms_per_step": round(grpA, 4), "alg_bytes_per_px": bytesA,
                "achieved_gbs": round(bytesA * px / (grpA * 1e-3) / 1e9, 1),
                "frac": round(bytesA * px / (grpA * 1e-3) / 1e9 / peak, 4)}

    res = None
    if rank == 0:
        res = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, world),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_ms,
                    "h2d_gbs_per_rank": round(h2d / (e2e_ms * 1e-3) / 1e9, 1), "numa": numa,
                    "bound": "host->device copy of the step's inputs (%.2f GB per rank and step over PCIe; the kernels "
                             "of a step take %.1f ms, the copy %.1f ms)" % (h2d / 1e9, ms_per_step, e2e_ms)},
            "gpu_launches": gpu_launches, "clocks": clk, "loss": loss_val, "ohem": ohem, "hist_check": hist_check,
            "workloads": [aux_workload] if aux_workload else [],
            "roofline": roof, "kernels": per_kernel,
        }
    return res


# ---------------------------------------------------------------------------------------------
# CPU arms: the oracle's torch restatement of the reference path on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_step(bt):
    """One pass of the SAME path with the reference's torch ops on CPU tensors (oracle/torch_ref.py)."""
    from oracle import label_space as ls, torch_ref as tr
    ids = bt["ids"]
    ids_t = torch.tensor(ids, dtype=torch.int32)
    labels = torch.empty(bt["raw"].shape, dtype=torch.int64)
    for d, s, e in dataset_slices(ids):
        labels[s:e] = torch.from_numpy(ls.lut_gather(bt["raw"][s:e].numpy(), bt["luts"][d]).astype(np.int64))
    x = bt["x"].detach().requires_grad_(True)
    loss = tr.multi_dataset_seg_loss(x, labels, ids_t, bt["graphs"], 0.4)
    loss.backward()
    mious = []
    for d, s, e in dataset_slices(ids):
        h = ls.confusion(labels[s:e].numpy(), bt["pred"][s:e].numpy(), bt["n_cats"][d])
        mious.append(ls.ious_miou(h)[1])
    return float(loss.detach()), mious


def run_eager_gpu(args, local_rank):
    """Context number (SURVEY §8d): the reference's torch ops on the same B200, full batch, device-resident."""
    dev = torch.device(f"cuda:{local_rank}")
    bt = make_batch(args.workload, dev, 1234)
    bt["graphs"] = [g.to(dev) for g in bt["graphs"]]
    luts = [torch.from_numpy(l).to(dev) for l in bt["luts"]]
    ids = bt["ids"]
    ids_t = torch.tensor(ids, dtype=torch.int32, device=dev)
    from oracle import torch_ref as tr

    def step():
        labels = torch.empty(bt["raw"].shape, dtype=torch.int64, device=dev)
        for d, s, e in dataset_slices(ids):
            labels[s:e] = luts[d][bt["raw"][s:e].long()].long()
        x = bt["x"].detach().requires_grad_(True)
        loss = tr.multi_dataset_seg_loss(x, labels, ids_t, bt["graphs"], 0.4)
        loss.backward()
        mious = []
        for d, s, e in dataset_slices(ids):
            c = bt["n_cats"][d]
            keep = labels[s:e] != 255
            h = torch.bincount(labels[s:e][keep] * c + bt["pred"][s:e][keep], minlength=c * c).view(c, c).double()
            iou = h.diag() / (h.sum(0) + h.sum(1) - h.diag())
            mious.append(torch.nanmean(iou))
        return loss.detach(), torch.stack(mious)

    step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 3
    e0.record()
    for _ in range(n):
        out = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    px = len(ids) * bt["H"] * bt["W"]
    return {"value": px / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "loss": float(out[0]),
            "what": "oracle/torch_ref.py (einsum -> F.interpolate -> CrossEntropyLoss(none) -> OHEM) + torch.bincount, "
                    "PyTorch eager on this GPU, device-resident inputs"}


def cpu_sample_images(workload):
    ids = WORKLOADS[workload][2]
    if workload in ("cfg3", "cfg2"):
        # one full-resolution image of EVERY dataset: the sample's mean class count (cfg3: 64) matches the
        # batch's (61.2), so pixels/s of the sample is representative of the whole batch
        return [ids.index(d) for d in sorted(set(ids))]
    return list(range(len(ids)))


def run_cpu(args, steps, warmup):
    torch.set_num_threads(os.cpu_count())
    images = cpu_sample_images(args.workload)
    bt = make_batch(args.workload, "cpu", 1234, images=images, logits=args.logits)
    px = len(images) * bt["H"] * bt["W"]
    for _ in range(warmup):
        cpu_step(bt)
    t0 = time.perf_counter()
    for _ in range(steps):
        cpu_step(bt)
    dt = (time.perf_counter() - t0) / steps
    return {"value": px / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"images {images} of the {args.workload} batch at full resolution ({px} px per step), "
                      f"oracle/torch_ref.py + numpy bincount (the reference's own torch ops), fp32, "
                      f"{warmup} warm-up + {steps} timed step(s) of {dt:.2f} s"}, dt


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        if rank != 0:
            return
        # exactly the steps and warm-up asked for; one step = the bounded sample run_cpu names (~3 s on 16 cores),
        # so the driver's --steps 20 --warmup 5 is about 75 s
        cb, dt = run_cpu(args, steps=max(1, args.steps), warmup=max(0, args.warmup))
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args, args.gpus),
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the mdseg hot path has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    res = run_ours(args, rank, world, local_rank)
    if _AFFINITY_BEFORE:  # every thread of the process (OpenMP workers created meanwhile inherited the narrow mask)
        for tid in os.listdir("/proc/self/task"):
            try:
                os.sched_setaffinity(int(tid), _AFFINITY_BEFORE[0])
            except OSError:
                pass
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            cb, _ = run_cpu(args, steps=2, warmup=1)
            res["cpu_baseline"] = cb
        else:
            res["cpu_baseline"] = None
        if args.eager_gpu and world == 1:
            torch.cuda.empty_cache()
            res["reference_eager_gpu"] = run_eager_gpu(args, local_rank)
        print(json.dumps(res))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
