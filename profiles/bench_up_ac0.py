"""Side benchmark: the BiSeNet heads' align_corners=False up-sampling + OhemCELoss, forward + backward, at every
head shape of BiSeNetV2 on BASELINE cfg1 (2x19x512x1024) and cfg4 (16x171x640x640): main x8, aux x2, x4, x8, x16
(the main head and the x8 aux head share a shape).

    python profiles/bench_up_ac0.py [--out FILE.jsonl] [--reps 7]

Route A (what runs without the fusion): F.interpolate(..., mode='bilinear', align_corners=False) + ops.ohem_ce.
Route B: ops.up_ohem_ce(..., align_corners=False).  A and B alternate in one process, CUDA events around each
forward + backward, 256 MB of L2 flush before every timed pass, median of the repetitions.  One JSON line per
measurement on stdout and in --out; the first line names the card and its power limit.  `ex2_floor_ms` is
arithmetic, not a measurement: 2 N H W C exponentials (forward and backward) at 16 per clock and SM, 148 SMs,
at the card's maximum SM clock."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from mdseg_b200 import ops  # noqa: E402

DEV = "cuda:0"
CFGS = {"cfg1": (2, 19, 512, 1024), "cfg4": (16, 171, 640, 640)}
FACTORS = (2, 4, 8, 16)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_up_ac0 measures on a CUDA device; none is visible")
    out = open(args.out, "w") if args.out else None

    def emit(**kv):
        line = json.dumps(kv)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    smi = q.stdout.strip().splitlines()[0] if q.stdout else None
    emit(card=torch.cuda.get_device_name(0), nvidia_smi=smi)
    try:
        clk_mhz = float(smi.split(",")[2].split()[0])
    except Exception:
        clk_mhz = None
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    thresh = ops.neg_log(0.7)

    for cfg, (N, C, H, W) in CFGS.items():
        for f in FACTORS:
            for dt in (torch.float32, torch.bfloat16):
                g = torch.Generator(device=DEV).manual_seed(f)
                src = (torch.randn(N, C, H // f, W // f, generator=g, device=DEV) * 3).to(dt).requires_grad_(True)
                lb = torch.randint(0, C, (N, H, W), generator=g, device=DEV)
                lb[torch.rand(N, H, W, generator=g, device=DEV) < 0.05] = 255

                def route_a():
                    src.grad = None
                    up = F.interpolate(src, size=(H, W), mode="bilinear", align_corners=False)
                    loss = ops.ohem_ce(up, lb, thresh)
                    loss.backward()
                    return loss

                def route_b():
                    src.grad = None
                    loss = ops.up_ohem_ce([src], lb, None, thresh, align_corners=False)[0]
                    loss.backward()
                    return loss

                la, lbv = float(route_a()), float(route_b())
                route_a()
                ga = src.grad.float().clone()
                route_b()
                gb = src.grad.float()
                grad_rel = float((ga - gb).abs().max() / ga.abs().max().clamp_min(1e-30))
                del ga, gb
                for _ in range(2):
                    route_a()
                    route_b()
                times = {"A": [], "B": []}
                for _ in range(args.reps):
                    for name, fn in (("A", route_a), ("B", route_b)):
                        flush.fill_(1)
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        fn()
                        e1.record()
                        torch.cuda.synchronize()
                        times[name].append(e0.elapsed_time(e1))
                med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
                floor = 2.0 * N * H * W * C / (16 * sms * clk_mhz * 1e6) * 1e3 if clk_mhz else None
                emit(cfg=cfg, head=("main x8 / aux x8" if f == 8 else f"aux x{f}"), shape=[N, C, H // f, W // f],
                     labels=[N, H, W], dtype=str(dt).replace("torch.", ""), route_a_ms=round(med["A"], 4),
                     route_b_ms=round(med["B"], 4), speedup=round(med["A"] / med["B"], 3),
                     route_a_all_ms=[round(t, 4) for t in times["A"]],
                     route_b_all_ms=[round(t, 4) for t in times["B"]],
                     ex2_floor_ms=None if floor is None else round(floor, 4),
                     route_b_over_ex2_floor=None if floor is None else round(med["B"] / floor, 3),
                     loss_a=la, loss_b=lbv, loss_rel_diff=abs(la - lbv) / abs(la), grad_rel_diff=grad_rel)
                del src, lb
                torch.cuda.empty_cache()
    if out:
        out.close()


if __name__ == "__main__":
    main()
