"""Side benchmark (not the headline): channels_last (NHWC) logits in the SEG-stage loss at the cfg3 shape
(16 x 358 x 256 x 512 unified logits, 1024 x 2048 uint8 labels, 7 datasets, column-one-hot graphs), fp32 and bf16.

Per dtype, forward + backward step time (median of CUDA-event timings after warm-up; every working set is far above
the 126 MB L2) for
  * the main head: NCHW input, channels_last input (mdseg_proj_fwd_nhwc / mdseg_proj_bwd_nhwc), and the copy route a
    channels_last model paid before: x.contiguous() -> NCHW call -> gradient .contiguous(channels_last);
  * the aux heads (up_ohem_ce over 7 per-dataset sources [16, C_d, 256, 512]): the same three;
  * the two NHWC projection kernels alone, with their algorithmic bytes as a fraction of the 6460 GB/s copy peak the
    project uses and of the 7.7 TB/s HBM3e data-sheet figure.
One JSON line per measurement on stdout; the first line names the card and its power limit."""
import ctypes as C
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from mdseg_b200 import native as N, ops  # noqa: E402

DEV = "cuda:0"
COPY_PEAK_GBS, DATASHEET_GBS = 6460.0, 7700.0
N_CATS = [19, 64, 37, 19, 26, 150, 133]
IDS = [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6]
C_UNI, h, w, H, W = 358, 256, 512, 1024, 2048
CL = torch.channels_last


def timed(fn, warmup=3, reps=9):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit(card=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)


def main_head(dt, graphs, labels, ids):
    g = torch.Generator(device=DEV).manual_seed(1)
    x = (torch.randn(len(IDS), C_UNI, h, w, generator=g, device=DEV) * 2.5).to(dt)
    xl = x.contiguous(memory_format=CL)
    th = ops.neg_log(0.4)

    def direct(t):
        def f():
            t.grad = None
            ops.mds_proj_ohem_ce(t, labels, ids, graphs, th).backward()
        return f

    def copy_route():
        xc = xl.detach().contiguous().requires_grad_(True)
        ops.mds_proj_ohem_ce(xc, labels, ids, graphs, th).backward()
        xl.grad = xc.grad.contiguous(memory_format=CL)

    xl.requires_grad_(True)
    x.requires_grad_(True)
    res = {"nchw": timed(direct(x)), "channels_last": timed(direct(xl)), "copy_route": timed(copy_route)}
    for k, v in res.items():
        emit(case=f"main head step {dt}", input=k, ms=round(v, 4))
    del x
    return xl.detach()


def aux_heads(dt, labels, ids):
    g = torch.Generator(device=DEV).manual_seed(2)
    srcs = [(torch.randn(len(IDS), c, h, w, generator=g, device=DEV) * 2.0).to(dt) for c in N_CATS]
    th = ops.neg_log(0.7)

    def direct(ts):
        def f():
            for t in ts:
                t.grad = None
            torch.nansum(ops.up_ohem_ce(ts, labels, ids, th)).backward()
        return f

    cl = [s.contiguous(memory_format=CL).requires_grad_(True) for s in srcs]
    nchw = [s.requires_grad_(True) for s in srcs]

    def copy_route():
        cs = [s.detach().contiguous().requires_grad_(True) for s in cl]
        torch.nansum(ops.up_ohem_ce(cs, labels, ids, th)).backward()
        for s, c in zip(cl, cs):
            s.grad = c.grad.contiguous(memory_format=CL)

    res = {"nchw": timed(direct(nchw)), "channels_last": timed(direct(cl)), "copy_route": timed(copy_route)}
    for k, v in res.items():
        emit(case=f"aux heads step {dt}", input=k, ms=round(v, 4))


def kernels(dt, xl, graphs, ids):
    tab, keep = ops._default_graphs.table(graphs)
    cmax = max(N_CATS)
    B, hw, e = len(IDS), h * w, xl.element_size()
    y = torch.empty(B, cmax, h, w, device=DEV)
    ymax = torch.empty(B, h, w, device=DEV)
    dx = torch.empty_like(xl)
    dy = torch.randn(B, cmax, h, w, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    ef = ops.err_flag(DEV)
    y_planes = sum(N_CATS[d] for d in IDS)  # the planes actually written / read

    def fwd():
        for _ in range(10):
            N.call("mdseg_proj_fwd_nhwc", xl.data_ptr(), ops._DT[dt], C.byref(tab), ids.data_ptr(), B, h, w,
                   y.data_ptr(), cmax, ymax.data_ptr(), ef.data_ptr(), s)

    def bwd():
        for _ in range(10):
            N.call("mdseg_proj_bwd_nhwc", dy.data_ptr(), None, cmax, C.byref(tab), ids.data_ptr(), B, h, w,
                   dx.data_ptr(), ops._DT[dt], s)

    for name, fn, nbytes in (("mdseg_proj_fwd_nhwc", fwd, B * hw * C_UNI * e + (y_planes + B) * hw * 4),
                             ("mdseg_proj_bwd_nhwc", bwd, y_planes * hw * 4 + B * hw * C_UNI * e)):
        ms = timed(fn) / 10
        gbs = nbytes / (ms * 1e-3) / 1e9
        emit(case=f"kernel {name} {dt}", ms=round(ms, 4), alg_bytes=nbytes,
             alg_B_per_label_px=round(nbytes / (B * H * W), 2), achieved_gbs=round(gbs, 1),
             frac_of_copy_peak_6460=round(gbs / COPY_PEAK_GBS, 4), frac_of_datasheet_7700=round(gbs / DATASHEET_GBS, 4))


def main():
    card()
    gen = torch.Generator().manual_seed(7)
    graphs = []
    for c in N_CATS:
        idx = torch.randint(0, c, (C_UNI,), generator=gen)
        idx[:c] = torch.arange(c)
        m = torch.zeros(c, C_UNI)
        m[idx, torch.arange(C_UNI)] = 1
        graphs.append(m.to(DEV))
    dg = torch.Generator(device=DEV).manual_seed(7)
    labels = torch.stack([torch.randint(0, N_CATS[d], (H, W), generator=dg, device=DEV) for d in IDS])
    labels[torch.rand(labels.shape, generator=dg, device=DEV) < 0.05] = 255
    labels = labels.to(torch.uint8)
    ids = torch.tensor(IDS, dtype=torch.int32, device=DEV)
    for dt in (torch.float32, torch.bfloat16):
        xl = main_head(dt, graphs, labels, ids)
        kernels(dt, xl, graphs, ids)
        del xl
        aux_heads(dt, labels, ids)
        torch.cuda.empty_cache()
    ops.check_errors(DEV)


if __name__ == "__main__":
    main()
