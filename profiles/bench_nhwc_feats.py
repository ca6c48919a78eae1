"""Side benchmark (not the headline): channels_last 16-bit features in the GNN stage at the cfg3 shape (16 x 512 x
256 x 512 features, 1024 x 2048 uint8 labels, 7 datasets, C_uni = 358, trainable dense graphs), bf16 and fp16.

Per dtype, forward + backward step time (median of CUDA-event timings after warm-up; the features alone are 2.15 GB,
far above the 126 MB L2) and the peak-memory growth of one step, for
  * the folded single loss (mds_head_proj_ohem_ce), the stacked hard / soft pair (mds_head_proj_ohem_ce_heads) and
    prototype_head forward + d feats + d proto;
  * each with (a) NCHW features, (b) channels_last features on the tc16 route with layout NHWC, (c) channels_last features
    through the copy route: feats.contiguous() -> NCHW call -> gradient .contiguous(channels_last);
and the three C-ABI calls of the folded loss alone (planar and pixel-major x, same operands).
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
N_CATS = [19, 64, 37, 19, 26, 150, 133]
IDS = [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6]
K, C_UNI, h, w, H, W = 512, 358, 256, 512, 1024, 2048
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


def peak(fn):
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def emit(**kw):
    print(json.dumps(kw), flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit(card=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)


def steps(dt, labels, ids):
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn(len(IDS), K, h, w, generator=g, device=DEV).to(dt)
    xl = x.contiguous(memory_format=CL)
    proto = (torch.randn(C_UNI, K, generator=g, device=DEV) * 0.05).requires_grad_(True)
    gs = [torch.rand(N_CATS[i % 7], C_UNI, generator=g, device=DEV).requires_grad_(True) for i in range(14)]
    dy = torch.randn(len(IDS), C_UNI, h, w, generator=g, device=DEV) * 1e-3
    th = ops.neg_log(0.4)
    routes = {
        "folded single": lambda t: ops.mds_head_proj_ohem_ce(t, proto, labels, ids, gs[:7], th).backward(),
        "stacked pair": lambda t: ops.mds_head_proj_ohem_ce_heads(t, proto, labels, ids, [gs[:7], gs[7:]], th).sum()
        .backward(),
        "prototype_head": lambda t: ops.prototype_head(t, proto).backward(dy),
    }
    x.requires_grad_(True)
    xl.requires_grad_(True)
    for name, run in routes.items():
        def direct(t):
            def f():
                for p in (t, proto, *gs):
                    p.grad = None
                run(t)
            return f

        def copy_route():
            for p in (xl, proto, *gs):
                p.grad = None
            xc = xl.detach().contiguous().requires_grad_(True)
            run(xc)
            xl.grad = xc.grad.contiguous(memory_format=CL)

        fns = {"a_nchw": direct(x), "b_channels_last": direct(xl), "c_copy_route": copy_route}
        for k, fn in fns.items():
            ms = timed(fn)
            mem = peak(fn)
            emit(case=f"{name} step {dt}", input=k, ms=round(ms, 4), peak_growth_gb=round(mem / 1e9, 3))
    return x.detach(), xl.detach(), gs


def calls(dt, x, xl, gs, ids):
    """The three C-ABI calls of the folded single loss, planar vs pixel-major, on the same operands."""
    n, cmax = 7, max(N_CATS)
    B, hw = len(IDS), h * w
    W_d = [g.detach() @ torch.randn(C_UNI, K, device=DEV) * 0.05 for g in gs[:7]]
    wt, ptrs, ldb = ops._tc16_operands(W_d, dt)
    wtt, ptrs_t, ldb_t = ops._tc16_operands(W_d, dt, transpose=True)
    cds = (C.c_int * n)(*N_CATS)
    y = torch.empty(B, cmax, h, w, device=DEV)
    dy16 = (torch.randn(B, cmax, h, w, device=DEV) * 1e-3).to(dt)
    dx = torch.empty_like(x)
    dxl = torch.empty_like(xl)
    dG = torch.empty(n, cmax, K, device=DEV)
    nb = N.lib.mdseg_proj_bwd_graph_tc16_workspace_bytes(B, K, hw, cmax)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    d = ops._DT[dt]
    for lname, lay, xx, dd in (("NCHW", N.NCHW, x, dx), ("NHWC", N.NHWC, xl, dxl)):
        fns = {
            "proj_fwd_tc16": lambda: N.call("mdseg_proj_fwd_tc16", xx.data_ptr(), d, lay, B, K, hw, ptrs, ldb, cds, n,
                                            ids.data_ptr(), y.data_ptr(), cmax, s),
            "proj_bwd_tc16": lambda: N.call("mdseg_proj_bwd_tc16", dy16.data_ptr(), d, lay, B, cmax, hw, ptrs_t, ldb_t,
                                            K, n, ids.data_ptr(), dd.data_ptr(), d, s),
            "proj_bwd_graph_tc16": lambda: N.call("mdseg_proj_bwd_graph_tc16", dy16.data_ptr(), xx.data_ptr(), d, lay,
                                                  B, K, hw, cmax, ids.data_ptr(), n, dG.data_ptr(), ws.data_ptr(), nb, s),
        }
        for k, fn in fns.items():
            emit(case=f"call {dt}", entry=f"mdseg_{k}", layout=lname, ms=round(timed(fn, 3, 21), 4))


def main():
    assert torch.cuda.is_available(), "bench_nhwc_feats.py measures on the GPU"
    card()
    g = torch.Generator(device=DEV).manual_seed(7)
    labels = torch.stack([torch.randint(0, N_CATS[d], (H, W), generator=g, device=DEV) for d in IDS])
    labels[torch.rand(labels.shape, generator=g, device=DEV) < 0.05] = 255
    labels = labels.to(torch.uint8)
    ids = torch.tensor(IDS, dtype=torch.int32, device=DEV)
    for dt in (torch.bfloat16, torch.float16):
        x, xl, gs = steps(dt, labels, ids)
        calls(dt, x, xl, gs, ids)
        del x, xl, gs
        torch.cuda.empty_cache()
    ops.check_errors(DEV)


if __name__ == "__main__":
    main()
