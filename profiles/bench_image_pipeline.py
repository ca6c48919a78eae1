"""Side benchmark (SURVEY §8 f3): the image branch of the training transforms for one ltbgnn_7_datasets_snp batch —
28 decoded uint8 BGR images (1024 x 2048 x 3, 4 per dataset) -> INTER_LINEAR resize (scale 0.5 .. 2.0, times
1080 / 1024) -> zero pad -> 768 x 768 crop -> flip -> ColorJitter(0.4, 0.4, 0.4) -> ToTensor(mean, std), fp32, as ONE
gather kernel (ops.image_pipeline), NCHW and channels_last output; then image + label (TrainPipeline, both kernels).

Times are medians of CUDA events over 9 calls, with a 256 MB buffer written before each call so that neither the
sources (176 MB) nor the output (198 MB) are served from the 126 MB L2.  `call_ms` is the Python call (views built
and uploaded per call, as a training loop would), `kernel_ms` the C-ABI call on an uploaded view table.  Algorithmic
bytes = 12 B per output pixel + the distinct source bytes the crops touch.  CPU column: the reference's per-sample
chain (cv2.resize, np.pad, crop, flip, the ColorJitter tables and np.matmul, ToTensor) with real cv2 on ONE host
core, as a DataLoader worker runs it; decode excluded.  The first line names the card and its power limit."""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402
from mdseg_b200 import native as N, ops  # noqa: E402
from mdseg_b200.dropin.label_transform import TrainPipeline  # noqa: E402
from oracle import image_space as ims  # noqa: E402

DEV = "cuda:0"
B, Hs, Ws, SIZE = 28, 1024, 2048, (768, 768)
NORMS = [((0.3257, 0.3690, 0.3223), (0.2112, 0.2148, 0.2115)), ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))] * 4
NORMS = NORMS[:7]
HBM_DATASHEET_GBS = 7700.0


def emit(**kw):
    print(json.dumps(kw), flush=True)


def timed(fn, flush, reps=9):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def touched_source_bytes(plans):
    n = 0
    for pl in plans:
        ys = np.arange(SIZE[0]) + pl["crop_y"] - pl["pad_top"]
        xs = np.arange(SIZE[1]) + pl["crop_x"] - pl["pad_left"]
        ys, xs = ys[(ys >= 0) & (ys < pl["im_h"])], xs[(xs >= 0) & (xs < pl["im_w"])]
        ry = ims._linear_taps(pl["im_h"], Hs, False)
        rx = ims._linear_taps(pl["im_w"], Ws, True)
        rows = np.unique(np.concatenate([ry[0][ys], ry[1][ys]]))
        cols = np.unique(np.concatenate([rx[0][xs], rx[1][xs]]))
        n += len(rows) * len(cols) * 3
    return n


def reference_chain(im_bgr, pl, mean, std):
    """lib/transform_cv2.py, per sample, with the draws of `pl`."""
    import cv2
    im = im_bgr[:, :, ::-1]
    im = cv2.resize(im, (pl["im_w"], pl["im_h"]))
    ph, pw = pl["pad_top"], pl["pad_left"]
    if ph > 0 or pw > 0:
        im = np.pad(im, ((ph, ph), (pw, pw), (0, 0)))
    im = im[pl["crop_y"]:pl["crop_y"] + SIZE[0], pl["crop_x"]:pl["crop_x"] + SIZE[1], :].copy()
    if pl["flip"]:
        im = im[:, ::-1, :]
    jt = pl["jitter"]
    im = np.array([i * jt["brightness"] for i in range(256)]).clip(0, 255).astype(np.uint8)[im]
    im = np.array([74 + (i - 74) * jt["contrast"] for i in range(256)]).clip(0, 255).astype(np.uint8)[im]
    r = jt["saturation"]
    M = np.float32([[1 + 2 * r, 1 - r, 1 - r], [1 - r, 1 + 2 * r, 1 - r], [1 - r, 1 - r, 1 + 2 * r]])
    im = np.clip(np.matmul(im.reshape(-1, 3), M).reshape(im.shape) / 3, 0, 255).astype(np.uint8)
    t = torch.from_numpy(im.transpose(2, 0, 1).astype(np.float32)).div_(255)
    return t.sub_(torch.as_tensor(mean)[:, None, None]).div_(torch.as_tensor(std)[:, None, None]).clone()


def main():
    assert torch.cuda.is_available(), "bench_image_pipeline.py measures on the GPU"
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    emit(card=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.stdout else None)
    rng = np.random.RandomState(1)
    raws = [rng.randint(0, 256, (Hs, Ws, 3)).astype(np.uint8) for _ in range(4)]
    srcs = [torch.from_numpy(raws[b % 4]).to(DEV) for b in range(B)]
    lbs = [torch.from_numpy(rng.randint(0, 34, (Hs, Ws)).astype(np.uint8)).to(DEV) for _ in range(B)]
    ids = [b // 4 for b in range(B)]
    luts = torch.from_numpy(rng.randint(0, 256, (7, 256)).astype(np.uint8)).to(DEV)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    tables = ops.to_tensor_tables(NORMS, DEV)
    px = B * SIZE[0] * SIZE[1]
    for fmt, name in ((torch.contiguous_format, "nchw"), (torch.channels_last, "channels_last")):
        pipe = TrainPipeline((0.5, 2.0), SIZE, luts=luts, norms=NORMS, memory_format=fmt)
        plans = pipe.plans([(Hs, Ws)] * B, np.random.RandomState(2))
        jts = [pl["jitter"] for pl in plans]
        alg = px * 12 + touched_source_bytes(plans)
        out = ops.image_pipeline(srcs, plans, SIZE, jitter=jts, norms=tables, norm_ids=ids, memory_format=fmt)
        want = ims.image_transform_chain(raws[5 % 4], plans[5], jts[5], *NORMS[ids[5]], SIZE, True)
        assert torch.equal(out[5].cpu(), torch.from_numpy(want))
        call_ms = timed(lambda: ops.image_pipeline(srcs, plans, SIZE, jitter=jts, norms=tables, norm_ids=ids,
                                                   memory_format=fmt), flush)
        # the C-ABI call alone, on a view table uploaded once
        table = ops.image_views(srcs, plans, jts, ids, tables.shape[0], True)
        layout = N.NHWC if fmt == torch.channels_last else N.NCHW
        kernel_ms = timed(lambda: N.call("mdseg_image_pipeline", table.data_ptr(), B, tables.data_ptr(), tables.shape[0],
                                         out.data_ptr(), layout, SIZE[0], SIZE[1], ops._stream()), flush)
        both_ms = timed(lambda: pipe(srcs, lbs, ids, plans=plans), flush)
        emit(case=f"{B} x (1024x2048x3 u8 BGR) -> 768x768 fp32", out=name, kernel_ms=round(kernel_ms, 4),
             call_ms=round(call_ms, 4), image_and_label_ms=round(both_ms, 4), out_Mpx=round(px / 1e6, 2),
             alg_bytes=alg, achieved_gbs_kernel=round(alg / kernel_ms / 1e6, 1),
             frac_of_datasheet_hbm=round(alg / kernel_ms / 1e6 / HBM_DATASHEET_GBS, 3))
    try:
        import cv2
    except ImportError:
        emit(cpu="not measured: cv2 is not installed on this host")
    else:
        cv2.setNumThreads(1)
        torch.set_num_threads(1)
        n = 8
        t0 = time.perf_counter()
        for b in range(n):
            ref = reference_chain(raws[b % 4], plans[b], *NORMS[ids[b]])
        cpu_ms = (time.perf_counter() - t0) / n * 1e3
        assert ref.shape == (3,) + SIZE
        emit(cpu="reference chain, real cv2 %s, one host core, decode excluded" % cv2.__version__,
             cpu_ms_per_sample=round(cpu_ms, 2), cpu_ms_per_batch_one_core=round(cpu_ms * B, 1))
    ops.check_errors(DEV)


if __name__ == "__main__":
    main()
