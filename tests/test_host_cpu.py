"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/mdseg.h declares,
the ctypes mirror matches the C structs, the drop-in modules import and parse configs, and the N > 1 logic
(image sharding, int64 histogram all-reduce, max-over-ranks timing) works under gloo with world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    src = open(os.path.join(ROOT, "include", "mdseg.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(mdseg_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from mdseg_b200 import native
    names = _declared_symbols()
    assert len(names) >= 25
    lib = ctypes.CDLL(native.LIB_PATH)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    unbound = [n for n in names if n not in native.SIGNATURES]
    assert not unbound, f"declared in mdseg.h but not bound in native.py: {unbound}"
    assert native.version() == 100


def test_struct_mirrors_match_the_c_layout(tmp_path):
    """sizeof() of every by-value struct as gcc sees it == the ctypes mirror."""
    from mdseg_b200 import native
    prog = tmp_path / "sz.c"
    prog.write_text('#include <stdio.h>\n#include "mdseg.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n",'
                    'sizeof(mdseg_ohem_state),sizeof(mdseg_src_table),sizeof(mdseg_sparse_graph),'
                    'sizeof(mdseg_graph_table),sizeof(mdseg_hist_table));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [ctypes.sizeof(native.OhemState), ctypes.sizeof(native.SrcTable), ctypes.sizeof(native.SparseGraph),
            ctypes.sizeof(native.GraphTable), ctypes.sizeof(native.HistTable)]
    assert got == want


def test_ops_refuse_cpu_tensors():
    from mdseg_b200 import ops
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.lut_remap(torch.zeros(4, dtype=torch.uint8), np.arange(256, dtype=np.uint8))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.ohem_ce(torch.zeros(1, 2, 2, 2), torch.zeros(1, 2, 2, dtype=torch.long), 0.35)


class DictConfiger:
    """Minimal stand-in for tools/configer.py:Configer (get / exists over nested dicts)."""

    def __init__(self, d):
        self.d = d

    def exists(self, *key):
        cur = self.d
        for k in key:
            if not isinstance(cur, dict) or k not in cur:
                return False
            cur = cur[k]
        return True

    def get(self, *key):
        cur = self.d
        for k in key:
            cur = cur[k]
        return cur


def test_dropin_modules_install_and_parse_configs():
    import json
    import mdseg_b200.dropin as dropin
    mods = dropin.install(extra=[("lib.loss.loss_cross_datasets", "loss_cross_datasets")])
    try:
        from lib.loss.ohem_ce_loss import MdsOhemCELoss, OhemCELoss
        from lib.class_remap import ClassRemap
        crit = OhemCELoss(0.7)
        assert abs(float(crit.thresh) - 0.35667494) < 1e-7 and crit.ignore_lb == 255
        cfg = json.load(open(os.path.join(ROOT, "tests", "golden", "test_test.json")))
        cfg.setdefault("loss", {}).setdefault("ignore_index", 255)
        cr = ClassRemap(DictConfiger(cfg))
        z = np.load(os.path.join(ROOT, "tests", "golden", "class_remap.npz"))
        for d in range(cr.n_datasets):
            assert np.array_equal(cr.getRemapMatrix(d).numpy(), z[f"test_d{d}_matrix"])
        assert [cr.IsSingleRemaplb(u) for u in range(cr.num_unify_classes)] == list(z["test_single_lbs"])
        assert MdsOhemCELoss(DictConfiger({"n_datasets": 2}), 0.4).n_datasets == 2
    finally:
        for name in mods:
            sys.modules.pop(name, None)


def test_shard_images_partitions_the_batch():
    from mdseg_b200.dist_utils import shard_images
    for n in (0, 1, 7, 16, 33):
        for w in (1, 2, 3, 8):
            parts = [list(shard_images(n, r, w)) for r in range(w)]
            assert sum(parts, []) == list(range(n))
            assert max(len(p) for p in parts) - min(len(p) for p in parts) <= 1


def test_shard_images_balanced_partitions_and_balances():
    """Cost-aware split for strong scaling: a partition with the same sizes as the contiguous one, identical on every
    rank, and on the cfg3 batch (class counts as costs) no rank above 1.4x the mean work (contiguous: 2.45x)."""
    from mdseg_b200.dist_utils import shard_images, shard_images_balanced
    n_cats = [19, 64, 37, 19, 26, 150, 133]
    ids = [0, 0, 0, 1, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6]
    costs = [n_cats[d] for d in ids]
    for w in (1, 2, 3, 4, 8, 16):
        parts = [shard_images_balanced(costs, r, w) for r in range(w)]
        assert sorted(sum(parts, [])) == list(range(len(costs)))
        assert [len(p) for p in parts] == [len(shard_images(len(costs), r, w)) for r in range(w)]
        assert all(p == sorted(p) for p in parts)
    work = lambda part: sum(costs[i] for i in part)
    mean = sum(costs) / 8
    assert max(work(shard_images_balanced(costs, r, 8)) for r in range(8)) <= 1.4 * mean
    assert max(work(list(shard_images(16, r, 8))) for r in range(8)) >= 2.4 * mean
    assert shard_images_balanced([], 0, 2) == [] and shard_images_balanced([5.0], 1, 2) == []


def _gloo_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    sys.path.insert(0, ROOT)
    from mdseg_b200 import dist_utils as du
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        assert du.world() == (rank, world)
        # every rank histograms its own shard of the images; the all-reduce must equal the global histogram
        g = torch.Generator().manual_seed(5)
        C, n_images, px = 7, 5, 4096
        label = torch.randint(0, C, (n_images, px), generator=g)
        pred = torch.randint(0, C, (n_images, px), generator=g)
        label[torch.rand(n_images, px, generator=g) < 0.1] = 255
        mine = list(du.shard_images(n_images, rank, world))
        hist = torch.zeros(C, C, dtype=torch.int64)
        for b in mine:
            keep = label[b] != 255
            hist += torch.bincount(label[b][keep] * C + pred[b][keep], minlength=C * C).view(C, C)
        hist[0, 0] += (1 << 40) + rank  # far beyond float32's exact range: the reduction must stay integer
        du.allreduce_hist(hist)
        keep = label != 255
        want = torch.bincount(label[keep] * C + pred[keep], minlength=C * C).view(C, C)
        want[0, 0] += world * (1 << 40) + sum(range(world))
        assert torch.equal(hist, want)
        with pytest.raises(TypeError):
            du.allreduce_hist(hist.float())
        # a step is as slow as the slowest rank; the whole-job rate counts every rank's pixels
        ms = du.max_over_ranks(10.0 + rank)
        assert ms == 10.0 + world - 1
        assert du.whole_job_rate(1000, world, ms) == 1000 * world / (ms * 1e-3)
        open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_world_size_2_gloo(tmp_path):
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_gloo_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert sorted(os.listdir(tmp_path)) == ["ok0", "ok1"]


def test_label_transform_planner_draws_the_reference_stream():
    """dropin.label_transform (host side of ops.label_pipeline) makes the same np.random draws in the same order as
    the restated RandomResizedCrop / RandomHorizontalFlip / ColorJitter sequence that tests/test_oracle_golden.py pins
    on the real lib/transform_cv2.py: same seed -> same plans, and the streams stay aligned over many samples."""
    import numpy as np
    from mdseg_b200.dropin.label_transform import LabelPipeline
    from oracle import label_space as ls
    shapes = [(96, 160), (1100, 1200), (1090, 1085), (300, 700), (64, 96), (2000, 1500)] * 3
    for scales, size, seed in (((0.5, 1.0), (64, 96), 1), ((0.03, 0.06), (64, 96), 2), ((0.75, 2.0), (256, 512), 3)):
        pipe = LabelPipeline(scales, size, p=0.5)
        got = pipe.plans(shapes, np.random.RandomState(seed))
        rng = np.random.RandomState(seed)
        for shape, g in zip(shapes, got):
            want = ls.plan_random_resized_crop(shape, scales, size, rng)
            want["flip"] = not (rng.random() < 0.5)
            for _ in range(3):
                rng.uniform(0.0, 1.0)
            assert g == want, (shape, g, want)


# ---- round 2: the drop-in really drops in (VERDICT r1 weak #2 / ADVICE high) -----------------------------------------
REFERENCE = os.environ.get("MDSEG_REFERENCE_ROOT", "")
needs_reference = pytest.mark.skipif(not REFERENCE or not os.path.isdir(os.path.join(REFERENCE, "lib")),
                                     reason="needs a checkout of the reference project under $MDSEG_REFERENCE_ROOT")

_TRAINER_IMPORTS = """
import sys, types, torch
sys.dont_write_bytecode = True
sys.path.insert(0, {root!r}); sys.path.insert(0, {ref!r})
tm, tmm, tml = types.ModuleType('timm'), types.ModuleType('timm.models'), types.ModuleType('timm.models.layers')
tml.trunc_normal_ = torch.nn.init.trunc_normal_   # the one name of `timm` the loss modules import (not installed here)
sys.modules.update({{'timm': tm, 'timm.models': tmm, 'timm.models.layers': tml}})
import mdseg_b200.dropin as dropin
dropin.install({install_args})
# tools/train_ltbgnn_all_datasets_snp.py:24,28,29 == tools/eval_snp.py:24,28,29, verbatim
from lib.loss.ohem_ce_loss import OhemCELoss
from lib.loss.loss_cross_datasets import CrossDatasetsLoss, CrossDatasetsCELoss, CrossDatasetsCELoss_KMeans, CrossDatasetsCELoss_CLIP, CrossDatasetsCELoss_GNN, CrossDatasetsCELoss_AdvGNN
from lib.class_remap import ClassRemap
# tools/train_amp.py:27 and lib/loss/loss_cross_datasets.py:6,12
from lib.loss.ohem_ce_loss import OhemCELoss, MdsOhemCELoss, MdsOhemNLLPlusLoss
from lib.class_remap import ClassRemap, ClassRemapOneHotLabel
import lib.loss.loss_cross_datasets as L
native = 'mdseg_b200.dropin'
assert OhemCELoss.__module__.startswith(native) and MdsOhemNLLPlusLoss.__module__.startswith(native)
assert ClassRemap.__module__.startswith(native)
assert L.OhemCELoss is OhemCELoss and L.MdsOhemNLLPlusLoss is MdsOhemNLLPlusLoss and L.ClassRemap is ClassRemap
print(CrossDatasetsCELoss_AdvGNN.__module__, CrossDatasetsCELoss.__module__, CrossDatasetsLoss.__module__, L.__name__)
"""


@needs_reference
@pytest.mark.parametrize("which", ["all_three", "leaf_modules_only"])
def test_install_then_the_trainers_import_lines(which, tmp_path):
    """After install() the reference's own import lines work — both with the loss module aliased (native
    CrossDatasetsCELoss*, the rest passed through) and with only the two leaf modules aliased (the reference's own
    lib/loss/loss_cross_datasets.py then imports MdsOhemNLLPlusLoss etc. from the drop-in, :6)."""
    args = "" if which == "all_three" else "only=['lib.loss.ohem_ce_loss', 'lib.class_remap']"
    code = _TRAINER_IMPORTS.format(root=ROOT, ref=REFERENCE, install_args=args)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    adv, ce, legacy, modname = r.stdout.split()
    if which == "all_three":
        assert adv.startswith("mdseg_b200.dropin") and ce.startswith("mdseg_b200.dropin")
        assert legacy.startswith("_mdseg_reference.")          # passed through from the reference's own file
    else:
        assert adv == ce == legacy == "lib.loss.loss_cross_datasets" == modname


@needs_reference
def test_reference_methods_run_on_the_dropin_classremap(tmp_path):
    """lib/test/test_class_remap.py:43-95 (the reference's own MultiProtoRemapping test body, CPU tensors) against the
    drop-in ClassRemapOneHotLabel: the method is the reference's, grafted onto the drop-in instance."""
    code = f"""
import sys, torch
sys.dont_write_bytecode = True
sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {REFERENCE!r})
import importlib.util
spec = importlib.util.spec_from_file_location('ref_class_remap', {REFERENCE!r} + '/lib/class_remap.py')
ref = importlib.util.module_from_spec(spec); spec.loader.exec_module(ref)
import mdseg_b200.dropin as dropin
dropin.install()
from lib.class_remap import ClassRemapOneHotLabel
from tools.configer import Configer
cfg = Configer(configs={REFERENCE!r} + '/configs/test/test.json')
ours, theirs = ClassRemapOneHotLabel(cfg), ref.ClassRemapOneHotLabel(cfg)
labels = torch.tensor([[2, 0, 0, 0], [2, 1, 1, 1], [2, 2, 1, 2], [0, 0, 0, 2]]).unsqueeze(0)
embed = torch.tensor([[[-0.1, 0.9], [0.9, 0.1]], [[-0.8, 0.2], [-0.1, 0.9]]]).unsqueeze(0).contiguous().view(-1, 2)
queue = torch.tensor([[[-1, 0], [0.9, 0.1], [-0.1, 1], [0, -1]], [[-0.9, 0.1], [1, 0], [0, 1], [-0.1, -1.9]]])
proto = torch.mm(embed, queue.view(-1, 2).T)
proto_logits = torch.zeros_like(proto)
for i in range(2):
    proto_logits[:, i::2] = proto[:, i * 4:(i + 1) * 4]
a = ours.MultiProtoRemapping(labels, proto_logits, 0)
b = theirs.MultiProtoRemapping(labels, proto_logits, 0)
assert all(torch.equal(x, y) for x, y in zip(a, b))
assert ours.getAnyClassRemap(2, 0) == theirs.getAnyClassRemap(2, 0) == [2, 3]
print('ok')
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr[-2000:]


def test_dropin_superset_without_a_reference_checkout(tmp_path):
    """No checkout on sys.path: the native names work, a passed-through name raises an AttributeError that says why."""
    code = f"""
import sys
sys.path.insert(0, {ROOT!r})
import mdseg_b200.dropin as dropin
dropin.install()
from lib.loss.ohem_ce_loss import OhemCELoss, MdsOhemCELoss, MdsOhemNLLPlusLoss
from lib.loss.loss_cross_datasets import CrossDatasetsCELoss, CrossDatasetsCELoss_GNN, CrossDatasetsCELoss_AdvGNN, LabelToOneHot
import lib.loss.loss_cross_datasets as L
try:
    L.CrossDatasetsLoss
except AttributeError as e:
    assert 'pass-through is unavailable' in str(e), e
    print('ok')
"""
    env = {k: v for k, v in os.environ.items() if k != "MDSEG_REFERENCE_ROOT"}
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path, env=env)
    assert r.returncode == 0 and r.stdout.strip() == "ok", r.stderr[-2000:] + r.stdout


def test_bench_reference_arm_contract_and_no_cpu_fallback():
    """bench.py --impl reference (the CPU arm the driver runs beside ours) prints ONE JSON line with the contract's keys,
    the steps it actually timed and the GPU arm's config object; without a CUDA device our arm refuses to run instead of
    falling back to the CPU."""
    import json
    import subprocess
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                        "--steps", "2", "--warmup", "1"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["name"] == "tiny" and "workload" in d["config"] and "model" not in d["config"]
    if not __import__("torch").cuda.is_available():
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "1"],
                           capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_bench_steps_and_dump_outputs(tmp_path):
    """--steps is the number of timed steps, so fewer than one is refused.  dump_outputs() stores integers as float64
    and the rest as float32, and keeps an array above DUMP_MAX_ELEMS as the same sorted sample of positions in every
    run."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    code = f"""
import sys, torch
sys.path.insert(0, {ROOT!r})
import bench
n = bench.DUMP_MAX_ELEMS + 1000
for d in ("a", "b"):
    bench.dump_outputs({str(tmp_path)!r} + "/" + d, {{"big": torch.arange(n, dtype=torch.float32).reshape(8, -1),
                                                      "hist": torch.arange(6).view(2, 3) << 40,
                                                      "half": torch.ones(3, dtype=torch.bfloat16), "none": None}})
print(bench.DUMP_MAX_ELEMS)
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=tmp_path, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    cap = int(r.stdout.split()[-1])
    assert sorted(os.listdir(tmp_path / "a")) == ["big.npy", "half.npy", "hist.npy"]
    big = np.load(tmp_path / "a" / "big.npy")
    assert big.dtype == np.float32 and big.shape == (cap,)
    assert np.all(np.diff(big) > 0) and big[0] >= 0 and big[-1] < cap + 1000  # distinct positions, in order
    assert np.array_equal(big, np.load(tmp_path / "b" / "big.npy"))
    hist = np.load(tmp_path / "a" / "hist.npy")
    assert hist.dtype == np.float64 and np.array_equal(hist, (np.arange(6).reshape(2, 3) << 40).astype(np.float64))
    assert np.load(tmp_path / "a" / "half.npy").dtype == np.float32
