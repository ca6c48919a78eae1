"""CPU: the oracle against the reference's known answers and against outputs of the real reference
modules (tests/golden/*.npz, see make_golden.py).  This is what 'pins' the oracle (SURVEY.md §8c)."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from oracle import f64, label_space as ls, torch_ref as tr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_kat_crossdatasets_celoss(golden):
    """lib/loss/test/test_loss_cross_datasets.py:118-145 — exact float equality with 5.106813430786133."""
    z = golden("kat_crossdatasets_celoss.npz")
    mats = [torch.from_numpy(z["matrix0"]), torch.from_numpy(z["matrix1"])]
    # the matrices are what ClassRemap builds from configs/test/test.json:26-36
    assert np.array_equal(z["matrix0"], ls.remap_matrix({0: [0], 1: [1], 2: [2, 3]}, 3, 4))
    assert np.array_equal(z["matrix1"], ls.remap_matrix({0: [3], 1: [2], 2: [1], 3: [0]}, 4, 4))
    loss = tr.remap_matrix_ce_loss(torch.from_numpy(z["logits"]), torch.from_numpy(z["labels"]),
                                   torch.from_numpy(z["ids"]), mats)
    assert float(loss) == 5.106813430786133 == float(z["loss"])
    # intermediate tensors of the reference test (:128-140)
    r0 = tr.project(torch.from_numpy(z["logits"][:1]), mats[0])
    assert r0.permute(0, 2, 3, 1).tolist() == [[[[1, 2, 7], [0, 1, 5]], [[2, 3, 5], [3, 0, 3]]]]
    r1 = tr.project(torch.from_numpy(z["logits"][1:]), mats[1])
    assert r1.permute(0, 2, 3, 1).tolist() == [[[[0, 2, 1, 3], [0, 1, 4, 2]], [[2, 0, 1, 3], [1, 3, 4, 2]]]]


def test_is_single_remap_lb_kat():
    """lib/test/test_class_remap.py:12-18 on configs/test/test_isSingleRemaplb.json (fixture restated here:
    class_remap1 = {0:[0],1:[1],2:[2,3]}, class_remap2 = {0:[3],1:[2],2:[1],3:[0]} -> lb 1 single)."""
    remaps = [{0: [0], 1: [1], 2: [2, 3]}]
    assert ls.is_single_remap_lb(remaps, 1) is True
    assert ls.is_single_remap_lb(remaps, 3) is False


@pytest.mark.parametrize("tag,cfg,n_ds", [("test", "test_test.json", 2), ("cca", "test_cca.json", 3)])
def test_class_remap_golden(golden, tag, cfg, n_ds):
    """ClassRemap.{SingleSegRemapping, SegRemapping, ReverseSegRemap, getRemapMatrix} of the real reference."""
    z = golden("class_remap.npz")
    raw = json.load(open(os.path.join(ROOT, "tests", "golden", cfg)))
    remaps, max_nums = ls.parse_class_remap(raw, n_ds)
    for d in range(n_ds):
        lb = z[f"{tag}_d{d}_labels"]
        assert np.array_equal(ls.single_seg_remapping(lb, remaps[d]), z[f"{tag}_d{d}_single"])
        segs = ls.seg_remapping(lb, remaps[d], max_nums[d])
        assert np.array_equal(np.stack(segs), z[f"{tag}_d{d}_seg"])
        m = ls.remap_matrix(remaps[d], raw[f"dataset{d + 1}"]["n_cats"], raw["num_unify_classes"])
        assert np.array_equal(m, z[f"{tag}_d{d}_matrix"])
        pr = z[f"{tag}_d{d}_preds"]
        assert np.array_equal(ls.reverse_seg_remap(pr, remaps[d], d), z[f"{tag}_d{d}_reverse"])
        # ... and the LUT form the kernels consume gives the same maps
        lut = ls.single_seg_lut(remaps[d])
        clipped = np.where((lb >= 0) & (lb < 256), lb, 0)
        assert np.array_equal(np.where((lb >= 0) & (lb < 256), lut[clipped], 255), z[f"{tag}_d{d}_single"])
        for j, lut_j in enumerate(ls.seg_luts(remaps[d], max_nums[d])):
            assert np.array_equal(lut_j[clipped], z[f"{tag}_d{d}_seg"][j])
        assert np.array_equal(ls.reverse_seg_lut(remaps[d], d)[pr], z[f"{tag}_d{d}_reverse"])
    singles = np.array([ls.is_single_remap_lb(remaps, u) for u in range(raw["num_unify_classes"])])
    assert np.array_equal(singles, z[f"{tag}_single_lbs"])


@pytest.mark.parametrize("tag,cfg,n_ds", [("test", "test_test.json", 2), ("cca", "test_cca.json", 3)])
def test_multihot_golden(golden, tag, cfg, n_ds):
    """ClassRemapOneHotLabel.{SegRemapping, SingleSegRemappingOneHot} of the real reference (class_remap.py:239-276):
    the per-class restatement and the [256, C_uni] table form the kernel consumes."""
    z = golden("multihot.npz")
    raw = json.load(open(os.path.join(ROOT, "tests", "golden", cfg)))
    remaps, _ = ls.parse_class_remap(raw, n_ds)
    cu = raw["num_unify_classes"]
    for d in range(n_ds):
        lb = z[f"{tag}_d{d}_labels"]
        assert np.array_equal(ls.multihot_seg_remapping(lb, remaps[d], cu), z[f"{tag}_d{d}_multi"])
        assert np.array_equal(ls.multihot_seg_remapping(lb, remaps[d], cu, single_only=True), z[f"{tag}_d{d}_single"])
        assert np.array_equal(ls.multihot_table(remaps[d], cu)[lb].astype(bool), z[f"{tag}_d{d}_multi"])
        assert np.array_equal(ls.multihot_table(remaps[d], cu, single_only=True)[lb].astype(bool), z[f"{tag}_d{d}_single"])


@pytest.mark.parametrize("name", ["thresh", "topk", "allign"])
def test_ohem_golden(golden, name):
    """OhemCELoss(0.7) of the real reference: value, gradient, both branches and the all-ignore NaN."""
    z = golden("ohem_ce.npz")
    logits = torch.from_numpy(z[f"ohem_{name}_logits"]).requires_grad_(True)
    labels = torch.from_numpy(z[f"ohem_{name}_labels"])
    loss = tr.ohem_ce_loss(logits, labels, 0.7)
    if name == "allign":
        assert np.isnan(float(loss)) and np.isnan(z["ohem_allign_loss"])
        return
    assert float(loss) == float(z[f"ohem_{name}_loss"])
    (loss * 3.0).backward()
    assert np.array_equal(logits.grad.numpy(), z[f"ohem_{name}_dlogits"])
    # float64 ground truth agrees to fp32 accuracy
    mean, dl, loss_px, mask = f64.ohem_ce(z[f"ohem_{name}_logits"], z[f"ohem_{name}_labels"], tr.neg_log_thresh(0.7))
    assert abs(mean - float(loss)) <= 2e-6 * abs(mean)
    assert np.abs(3.0 * dl - z[f"ohem_{name}_dlogits"]).max() <= 2e-6 * np.abs(dl).max() * 3
    assert (mask.sum() > 0) and ((name == "topk") == (mask.sum() == (z[f"ohem_{name}_labels"] != 255).sum() // 16))


@pytest.mark.parametrize("name", ["sorted", "shuffled", "absent", "dense"])
def test_mds_golden(golden, name):
    """einsum + interpolate + MdsOhemCELoss(0.4) of the real reference (sorted / unsorted / absent dataset /
    dense graphs with grad)."""
    z = golden("mds.npz")
    x = torch.from_numpy(z[f"mds_{name}_x"]).requires_grad_(True)
    labels = torch.from_numpy(z[f"mds_{name}_labels"])
    ids = torch.from_numpy(z[f"mds_{name}_ids"])
    graphs = [torch.from_numpy(z[f"mds_{name}_graph{i}"]).requires_grad_(name == "dense") for i in range(3)]
    loss = tr.multi_dataset_seg_loss(x, labels, ids, graphs, 0.4)
    assert float(loss) == float(z[f"mds_{name}_loss"])
    scale = 1.0 if name == "dense" else 2.0
    (loss * scale).backward()
    assert np.array_equal(x.grad.numpy(), z[f"mds_{name}_dx"])
    ref = f64.multi_dataset(z[f"mds_{name}_x"], z[f"mds_{name}_labels"], z[f"mds_{name}_ids"],
                            [g.detach().numpy() for g in graphs], tr.neg_log_thresh(0.4), want_graph_grads=True)
    assert abs(ref["loss"] - float(loss)) <= 2e-6 * abs(ref["loss"])
    assert np.abs(scale * ref["dlogits_uni"] - z[f"mds_{name}_dx"]).max() <= 5e-6 * np.abs(ref["dlogits_uni"]).max() * scale
    if name == "dense":
        for i in range(3):
            assert np.array_equal(graphs[i].grad.numpy(), z[f"mds_dense_dgraph{i}"])
            assert np.abs(ref["dgraphs"][i] - z[f"mds_dense_dgraph{i}"]).max() <= 1e-5 * np.abs(ref["dgraphs"][i]).max()


def test_advgnn_seg_stage_golden(golden):
    """CrossDatasetsCELoss_AdvGNN (SEG stage, 7 datasets, dataset aux heads) of the real reference."""
    z = golden("advgnn_seg_stage.npz")
    n = len(z["n_cats"])
    x = torch.from_numpy(z["x"]).requires_grad_(True)
    aux = [torch.from_numpy(z[f"aux{i}"]).requires_grad_(True) for i in range(n)]
    graphs = [torch.from_numpy(z[f"graph{i}"]) for i in range(n)]
    total, main, aux_loss = tr.seg_stage_total_loss(x, aux, torch.from_numpy(z["labels"]), torch.from_numpy(z["ids"]),
                                                    graphs, float(z["aux_weight"]))
    assert float(total) == float(z["loss"]) and float(aux_loss) == float(z["aux_loss"])
    total.backward()
    assert np.array_equal(x.grad.numpy(), z["dx"])
    for i in range(n):
        assert np.array_equal(aux[i].grad.numpy(), z[f"daux{i}"])


def test_c_oracle_matches_numpy_and_torch():
    lib = ctypes.CDLL(os.path.join(ROOT, "oracle", "_build", "liboracle.so"))
    rng = np.random.default_rng(3)
    # LUT
    raw = rng.integers(0, 256, 10007, dtype=np.uint8)
    lut = rng.integers(0, 256, 256, dtype=np.uint8)
    out = np.empty_like(raw)
    lib.orc_lut_remap_u8(raw.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p),
                         lut.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(raw.size))
    assert np.array_equal(out, ls.lut_gather(raw, lut))
    # confusion
    C = 19
    lab = rng.integers(0, C, 5000).astype(np.int64)
    lab[rng.random(5000) < 0.1] = 255
    pred = rng.integers(0, C, 5000).astype(np.int64)
    hist = np.zeros((C, C), dtype=np.int64)
    lib.orc_confusion_i64.restype = ctypes.c_int64
    bad = lib.orc_confusion_i64(lab.ctypes.data_as(ctypes.c_void_p), pred.ctypes.data_as(ctypes.c_void_p), None,
                                hist.ctypes.data_as(ctypes.c_void_p), C, C, 255, ctypes.c_int64(lab.size))
    assert bad == 0 and np.array_equal(hist, ls.confusion(lab, pred, C))
    # upsample + CE per pixel, fp32 in ATen's order, against torch itself
    Cc, h, w, H, W = 7, 5, 6, 17, 22
    src = (rng.standard_normal((Cc, h, w)) * 3).astype(np.float32)
    labels = rng.integers(0, Cc, (H, W)).astype(np.int64)
    labels[0, :5] = 255
    loss = np.empty((H, W), dtype=np.float32)
    zbuf = np.empty(Cc, dtype=np.float32)
    lib.orc_up_ce_image_f32(src.ctypes.data_as(ctypes.c_void_p), Cc, h, w, labels.ctypes.data_as(ctypes.c_void_p), H, W,
                            255, loss.ctypes.data_as(ctypes.c_void_p), zbuf.ctypes.data_as(ctypes.c_void_p))
    want = tr.ce_none(tr.upsample(torch.from_numpy(src)[None], (H, W)), torch.from_numpy(labels)[None])[0].numpy()
    assert np.abs(loss - want).max() <= 4e-6
    lp64, _ = f64.ce_per_pixel(f64.upsample(src[None], H, W), labels[None])
    assert np.abs(loss - lp64[0]).max() <= 4e-6
    # nearest
    big = rng.integers(0, 200, (37, 53)).astype(np.int64)
    small = np.empty((9, 14), dtype=np.int64)
    lib.orc_nearest_i64(big.ctypes.data_as(ctypes.c_void_p), 37, 53, small.ctypes.data_as(ctypes.c_void_p), 9, 14)
    assert np.array_equal(small, ls.nearest_resize(big, (9, 14)))
    assert np.array_equal(small, tr.nearest_label(torch.from_numpy(big)[None], (9, 14))[0].numpy())


def test_f64_upsample_matches_torch_and_adjoint():
    rng = np.random.default_rng(5)
    x = rng.standard_normal((2, 3, 6, 7))
    up = f64.upsample(x, 23, 26)
    want = tr.upsample(torch.from_numpy(x).float(), (23, 26)).numpy()
    assert np.abs(up - want).max() <= 2e-6
    g = rng.standard_normal(up.shape)
    # <up(x), g> == <x, up^T(g)>
    assert abs((up * g).sum() - (x * f64.upsample_adjoint(g, 6, 7)).sum()) <= 1e-9 * abs((up * g).sum())


def test_confusion_miou_restatement():
    """evaluate.py:86-98 restated; cross-checked against a direct double loop on a tiny case."""
    lab = np.array([0, 1, 2, 255, 1, 1, 2, 0])
    pred = np.array([0, 2, 2, 1, 1, 0, 2, 0])
    h = ls.confusion(lab, pred, 3)
    want = np.zeros((3, 3), dtype=np.int64)
    for l, p in zip(lab, pred):
        if l != 255:
            want[l, p] += 1
    assert np.array_equal(h, want)
    ious, miou = ls.ious_miou(h)
    assert np.allclose(ious, [2 / 3, 1 / 3, 2 / 3]) and abs(miou - 5 / 9) < 1e-6
    ious, miou = ls.ious_miou(np.array([[3, 0], [0, 0]]))  # absent class -> NaN, skipped by nanmean
    assert np.isnan(ious[1]) and miou == 1.0
    with pytest.raises(ValueError):
        ls.confusion(np.array([5]), np.array([0]), 3)


# ---- evaluator tail pinned on the REAL evaluate.py (tests/golden/make_golden_eval.py) -----------------------
def _eval_case(z, tag):
    labels = [torch.from_numpy(z[f"{tag}_label{i}"].astype(np.int64)) for i in range(int(z[f"{tag}_n_batches"]))]
    calls = [[torch.from_numpy(z[f"{tag}_call{i}_head0"])] for i in range(int(z[f"{tag}_n_calls"]))]
    hists = [z[f"{tag}_hist{i}"] for i in range(int(z[f"{tag}_n_hists"]))]
    return labels, calls, hists


@pytest.mark.parametrize("tag,n_scales,flip,ori", [("v0", 6, True, True), ("c_ori", 2, True, True),
                                                   ("c_low", 1, False, False), ("absent", 1, False, True)])
def test_evaluator_restatement_against_real_evaluate_py(golden, tag, n_scales, flip, ori):
    """oracle.torch_ref.eval_probs / eval_preds / nearest_label + oracle.label_space.confusion / ious_miou replay
    the logits the real MscEvalV0 / MscEvalV0_Contrast saw and must give their np.bincount results and mIoU."""
    z = golden("evaluator.npz")
    labels, calls, hists = _eval_case(z, tag)
    per_batch = n_scales * (2 if flip else 1)
    assert len(calls) == per_batch * len(labels) and len(hists) == len(labels)
    total = None
    for b, lb in enumerate(labels):
        passes = [c[0] for c in calls[b * per_batch:(b + 1) * per_batch]]
        flips = [bool(flip and (i % 2)) for i in range(per_batch)]
        lab = lb.squeeze(1)
        if ori:
            size = tuple(lab.shape[-2:])
        else:
            size = tuple(passes[0].shape[-2:])
            lab = tr.nearest_label(lab, size)
            assert np.array_equal(lab.numpy(), ls.nearest_resize(lb.squeeze(1).numpy(), size))
        pred = tr.eval_preds(tr.eval_probs(passes, size, flips))
        C = passes[0].shape[1]
        h = ls.confusion(lab.numpy(), pred.numpy(), C)
        assert np.array_equal(h.reshape(-1), hists[b])
        total = h if total is None else total + h
    assert abs(ls.ious_miou(total)[1] - float(z[f"{tag}_miou"])) <= 1e-7


def test_autolink_rectangular_hist_against_real_evaluate_py(golden):
    """evaluate.py:582-640: [n_classes, n_cats_k] histograms against the other datasets' heads, row arg-max."""
    z = golden("evaluator.npz")
    n_cats, me = [19, 12, 36], 1
    nb = int(z["autolink_n_batches"])
    tot = {k: np.zeros((n_cats[me], n_cats[k]), dtype=np.int64) for k in range(3) if k != me}
    hi = 0
    for b in range(nb):
        lab = z[f"autolink_label{b}"].astype(np.int64).squeeze(1)
        for k in tot:
            lg = torch.from_numpy(z[f"autolink_call{b}_head{k}"])
            pred = tr.eval_preds(tr.eval_probs([lg], lab.shape[-2:]))
            h = ls.confusion(lab, pred.numpy(), n_cats[me], n_cats[k])
            assert np.array_equal(h.reshape(-1), z[f"autolink_hist{hi}"])
            hi += 1
            tot[k] += h
    assert hi == int(z["autolink_n_hists"])
    for k in range(3):
        want = z[f"autolink_argmax{k}"]
        got = np.arange(n_cats[me]) if k == me else tot[k].argmax(axis=1)
        assert np.array_equal(got, want)


def test_advgnn_gnn_stage_golden(golden):
    """CrossDatasetsCELoss_AdvGNN of the real reference in the GNN stage (tests/golden/make_golden_gnn_stage.py):
    prototype head, (hard, soft) graph pairs blended by max_rate, aux heads from the prototypes, orth + adj terms."""
    z = golden("advgnn_gnn_stage.npz")
    n_cats = [19, 64, 37, 19, 26, 150, 133]
    feats = torch.from_numpy(z["feats"]).requires_grad_(True)
    proto = torch.from_numpy(z["proto"]).requires_grad_(True)
    graphs = [torch.from_numpy(z[f"graph{i}"]).requires_grad_(True) for i in range(14)]
    tgt = [torch.from_numpy(z[f"target{i}"]) for i in range(7)]
    loss, orth, aux, adj = tr.gnn_stage_total_loss(feats, proto, graphs, torch.from_numpy(z["labels"].astype(np.int64)),
                                                   torch.from_numpy(z["ids"]), n_cats, 21000 / 60000, tgt)
    for got, key in ((loss, "loss"), (orth, "orth"), (aux, "aux"), (adj, "adj")):
        assert abs(float(got) - float(z[key])) <= 2e-6 * abs(float(z[key])), key
    loss.backward()
    assert np.abs(feats.grad.numpy() - z["dfeats"]).max() <= 1e-6 * np.abs(z["dfeats"]).max()
    assert np.abs(proto.grad.numpy() - z["dproto"]).max() <= 1e-6 * np.abs(z["dproto"]).max()
    for i in range(14):
        want = z[f"dgraph{i}"]
        got = graphs[i].grad.numpy() if graphs[i].grad is not None else np.zeros_like(want)
        assert np.abs(got - want).max() <= 1e-6 * max(np.abs(want).max(), 1e-30), i


def test_find_use_and_unuse_hist_against_real_evaluate_py(golden):
    """evaluate.py:1846-1866: prototype einsum -> upsample -> softmax -> argmax over C_uni -> [n_cats, C_uni] bincount."""
    z = golden("evaluator.npz")
    proto = torch.from_numpy(z["fuu_proto"])
    c_uni = int(z["fuu_c_uni"])
    for i, c in enumerate(z["fuu_n_cats"]):
        for b in range(2):
            lab = z[f"fuu_label{i}_{b}"].astype(np.int64).squeeze(1)
            logits = tr.project(torch.from_numpy(z[f"fuu_emb{i}_{b}"]), proto)
            pred = tr.eval_preds(tr.eval_probs([logits], lab.shape[-2:]))
            h = ls.confusion(lab, pred.numpy(), int(c), c_uni)
            assert np.array_equal(h.reshape(-1), z[f"fuu_hist{i}_{b}"])


# ---- label branch of the data pipeline, pinned on the real lib/transform_cv2.py + cv2 ---------------------------
def _label_pipeline_cases(z):
    for tag in ("crop", "pad", "wide"):
        n = int(z[f"{tag}_n"])
        yield (tag, int(z[f"{tag}_seed"]), tuple(float(v) for v in z[f"{tag}_scales"]),
               tuple(int(v) for v in z[f"{tag}_size"]), z[f"{tag}_lut"],
               [z[f"{tag}_raw{k}"] for k in range(n)], [z[f"{tag}_lb{k}"] for k in range(n)])


def test_label_transform_chain_against_real_transform_cv2(golden):
    """oracle.label_space.{plan_random_resized_crop, cv2_nearest_resize, label_transform_chain} against the output of
    RandomResizedCrop -> RandomHorizontalFlip -> ColorJitter -> ToTensor of the reference (real cv2.resize), several
    samples from one seeded np.random stream (tests/golden/make_golden_label_pipeline.py)."""
    z = golden("label_pipeline.npz")
    for tag, seed, scales, size, lut, raws, wants in _label_pipeline_cases(z):
        rng = np.random.RandomState(seed)  # np.random.seed(seed) seeds the same legacy generator
        for raw, want in zip(raws, wants):
            plan = ls.plan_random_resized_crop(raw.shape, scales, size, rng)
            plan["flip"] = not (rng.random() < 0.5)
            for _ in range(3):
                rng.uniform(0.0, 1.0)  # ColorJitter's three draws
            got = ls.label_transform_chain(raw, lut, plan, size)
            assert got.dtype == np.int64 and np.array_equal(got, want.astype(np.int64)), tag


def test_lb_map_gather_against_real_dataset_readers(golden):
    """lib/base_dataset.py:81-82 through the REAL reader classes of the seven ltbgnn_7_datasets_snp datasets
    (tests/golden/make_golden_lb_maps.py): oracle.label_space.lut_gather reproduces their __getitem__ label."""
    z = golden("lb_maps.npz")
    for i in range(7):
        lut = z[f"lb_map{i}"]
        assert lut.shape == (256,) and lut.dtype == np.uint8
        assert np.array_equal(ls.lut_gather(z["raw"], lut), z[f"label{i}"]), str(z["names"][i])


# ---- round 2: the restated NLLPlus / plain-CE drivers against the real reference classes (r2_losses.npz) ----------
@pytest.fixture
def recorded_threads():
    """The nll_* fixtures were recorded with 8 intra-op threads.  ATen's CPU softmax over a non-last dim takes its
    vectorised or its scalar exp depending on where the per-thread chunks end, so the fp32 bits of the softmax (and of
    the gradients through -log of its projection) follow the thread count: the exact comparison holds at 8 threads."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


@pytest.mark.parametrize("name", ["thresh", "topk", "dense", "absent"])
def test_torch_ref_nll_plus_matches_reference(golden, recorded_threads, name):
    from oracle import torch_ref as tr
    z = golden("r2_losses.npz")
    x = torch.from_numpy(z[f"nll_{name}_x"]).requires_grad_(True)
    graphs = [torch.from_numpy(z[f"nll_{name}_graph{i}"]).requires_grad_(name == "dense") for i in range(3)]
    labels, ids = torch.from_numpy(z[f"nll_{name}_labels"]), torch.from_numpy(z[f"nll_{name}_ids"])
    loss = tr.mds_ohem_nll_plus_loss(x, labels, graphs, ids, 3, float(z[f"nll_{name}_thresh"]))
    (loss * 1.5).backward()
    assert float(loss) == float(z[f"nll_{name}_loss"])
    assert np.array_equal(x.grad.numpy(), z[f"nll_{name}_dx"])


def test_torch_ref_plain_ce_drivers_match_reference(golden):
    from oracle import torch_ref as tr
    z = golden("r2_losses.npz")
    x, lb, ids = torch.from_numpy(z["ce_x"]), torch.from_numpy(z["ce_labels"]), torch.from_numpy(z["ce_ids"])
    import make_golden_r2 as mk
    mats = []
    for d in range(3):
        m = torch.zeros(mk.N_CATS[d], mk.C_UNI)
        for k, v in mk.REMAP[d].items():
            m[int(k), v] = 1
        mats.append(m)
    assert float(tr.cross_datasets_ce_mean(x, lb, ids, mats, upsample_to_labels=False)) == float(z["ce_loss"])
