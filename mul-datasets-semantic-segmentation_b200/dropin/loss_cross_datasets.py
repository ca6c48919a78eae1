"""Drop-in for lib/loss/loss_cross_datasets.py: ``CrossDatasetsCELoss_AdvGNN`` (:812-1138) — the loss class the
``ltbgnn_*`` configs select with ``loss.type = "Adv_GNN"`` — in every stage the trainer calls it in, plus
``CrossDatasetsCELoss`` (:303-347), ``CrossDatasetsCELoss_CLIP`` (:662-712) and ``CrossDatasetsCELoss_GNN`` (:714-776)
on the same fused kernels.  Every other name of the reference module (``CrossDatasetsLoss``,
``CrossDatasetsCELoss_KMeans``, ``CrossDatasetsCELoss_AdvGNN_ce`` ...) is passed through from the reference's own file
(``_reference.py``), so the trainers' import line (tools/train_ltbgnn_all_datasets_snp.py:28) works unchanged.

``forward(preds, target, dataset_ids, is_adv=True, init_gnn_stage=False) -> (loss, orth_loss, aux_loss, adj_loss)``

What runs where:
  * the per-pixel work (SURVEY.md §8 rows a5-a10) goes through libmdseg_b200.so:
      - SEG stage (is_adv=False, 0/1 graphs): projection + bilinear up-sampling + CE + one OHEM selection over the
        batch from the LOW-resolution unified logits (:1006-1007, :1074), aux heads from ``preds['aux']`` (:1051-1056);
        channels_last ``preds['seg']`` / ``preds['aux']`` (a model run with memory_format=torch.channels_last) are
        taken as they are, without a layout copy, and get channels_last gradients;
      - GNN stage (is_adv=True, trainable soft / hard graph pairs): the same fused loss once per graph set, blended
        by ``max_rate`` (:1063-1071), with gradients to the logits AND to every ``bi_graphs[i]`` (tcgen05 split-K
        ``d bi_graph``); aux heads from the dataset prototypes (:941-951, :1044-1048) through the fused
        up-sample + OhemCE(0.7) kernels; channels_last bf16 / fp16 features (``preds['seg']``, K % 8 == 0) are taken as
        they are by the prototype head and the folded / dense-graph losses and get a channels_last gradient (the
        ``feats.index_select`` rows of the aux prototypes are a gathered copy either way);
  * the prototype contractions ``einsum('bchw,nc->bnhw', feats, unify_prototype[...])`` (:950, :961, :971) — the
    producer of the unified logits, SURVEY §8 f2 — run on the tcgen05 tensor cores.  With ``FOLD_PROTOTYPES`` (the
    default) the unified head and the bipartite projection behind it are ONE contraction with
    ``bi_graphs[i] @ unify_prototype`` (``ops.mds_head_proj_ohem_ce``): the product is associative, so the
    ``[B, C_uni, h, w]`` unified logits and their gradient never exist; with the switch off the head is its own GEMM
    (``ops.prototype_head``: forward, d feats and the split-K d prototype) in front of the projection, operation by
    operation as the reference.  The aux heads (:950) always use ``ops.prototype_head``; only the GridSplit variant
    (:779-809) keeps the library einsum (its backward masks the unified-logit gradient per class);
  * the graph regularisers (orth / spa / max-enc / adj MSE, init-stage graph and prototype MSE, adversarial BCE /
    MSE terms) act on ``[C_ds, C_uni]``-sized tensors; they are restated with the same torch ops.

Differences a caller can observe: dataset presence is read from ``dataset_ids`` once per call (one small D2H copy
when the ids live on the GPU; the reference synchronises through ``.any()`` / boolean indexing ≥ 2·n_datasets
times); ``if aux_loss:`` / ``if orth_loss:`` / ``if adj_loss:`` truthiness tests (host syncs; skipping a term that is
exactly 0) became ``is not None`` (adding the zero); ``torch.isnan(loss)`` (:1076) is applied with ``torch.where``.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

from .. import ops
from . import _reference
from .class_remap import ClassRemap, ClassRemapOneHotLabel  # noqa: F401  (configs name them: eval(class_remaper))
from .ohem_ce_loss import MdsOhemCELoss, MdsOhemNLLPlusLoss, OhemCELoss  # noqa: F401


# einsum(einsum(feats, prototypes), bi_graph) evaluated as einsum(feats, bi_graph @ prototypes): see ops.fold_prototypes.
# Module-level so that a run can be switched back to the reference's operation order (tests exercise both).
FOLD_PROTOTYPES = True

# Non-trainable bi_graphs are copied to the host once per tensor object to build their index lists (ops.BipartiteGraphs).
# A trainer whose SEG-stage graphs are 0/1 with at most one 1 per column AND rebuilt as new tensors every iteration can
# set this to True: the lists are then built on the device without a copy, and a graph of another kind raises at the next
# ops.check_errors().  Off by default because detached soft graphs are legal inputs of these classes.
ASSUME_ONEHOT01_GRAPHS = False


def _cfg(configer, *key, default=None):
    try:
        if hasattr(configer, "exists") and not configer.exists(*key):
            return default
        return configer.get(*key)
    except (KeyError, TypeError):
        return default


def LabelToOneHot(LabelVector, nClass, ignore_index=-1):
    """:18-26 — bool [len, nClass] one-hot of a 1-D label vector (rows of ignored labels stay empty)."""
    out = torch.zeros(len(LabelVector), nClass, dtype=torch.bool, device=LabelVector.device)
    keep = LabelVector != ignore_index
    out[keep, LabelVector[keep]] = 1
    return out


def _present_rows(dataset_ids, n_datasets):
    ids = torch.as_tensor(dataset_ids).reshape(-1).tolist()  # the one host read of a forward
    return [[b for b, v in enumerate(ids) if int(v) == i] for i in range(n_datasets)]


def _sum_present(per_dataset, present):
    """Sum of the entries of `per_dataset` [n_datasets] whose dataset has images (the reference skips the others,
    e.g. :333-334); None when the batch is empty."""
    idx = [i for i, rows in enumerate(present) if rows]
    if not idx:
        return None
    return per_dataset[torch.tensor(idx, device=per_dataset.device)].sum()


class CrossDatasetsCELoss(nn.Module):
    """:303-347 — remap-matrix projection of the unified logits (ClassRemap.getRemapMatrix) + plain cross-entropy
    (ignore 255) per dataset, summed over the datasets present.  Pinned by the reference's own known-answer test
    (lib/loss/test/test_loss_cross_datasets.py:118-145, 5.106813430786133)."""

    def __init__(self, configer=None):
        super().__init__()
        self.configer = configer
        self.n_datasets = self.configer.get('n_datasets')
        self.classRemapper = eval(self.configer.get('class_remaper'))(configer=self.configer)
        self.num_unify_classes = self.configer.get('num_unify_classes')
        self.num_prototype = _cfg(configer, 'contrast', 'num_prototype')
        self.temperature = _cfg(configer, 'contrast', 'temperature')
        self.with_mulbn = _cfg(configer, 'contrast', 'with_mulbn')
        self.reweight = _cfg(configer, 'loss', 'reweight')
        self.ignore_index = _cfg(configer, 'loss', 'ignore_index', default=255)
        self.n_cats = [configer.get('dataset' + str(i), 'n_cats') for i in range(1, self.n_datasets + 1)]
        self.CELoss = torch.nn.CrossEntropyLoss(ignore_index=255)  # kept for introspection only
        self._graph_cache = ops.BipartiteGraphs()
        self._matrices = None

    def forward(self, preds, target, dataset_ids, is_warmup=False):
        self.with_aux = self.configer.get('loss', 'with_aux')
        logits = preds['seg'][0] if self.with_aux else preds['seg']
        if self._matrices is None or self._matrices[0].device != logits.device:
            self._matrices = [self.classRemapper.getRemapMatrix(i).to(logits.device) for i in range(self.n_datasets)]
        present = _present_rows(dataset_ids, self.n_datasets)
        per_ds = ops.mds_proj_ce_mean(logits, target, dataset_ids, self._matrices, ignore=255, cache=self._graph_cache)
        return _sum_present(per_ds, present)


class CrossDatasetsCELoss_CLIP(nn.Module):
    """:662-712 — text-prototype head (optional), per-dataset projection (remap matrix or the dataset's text
    features), bilinear up-sampling to the label size and OhemCELoss(0.7) per dataset, summed."""

    def __init__(self, configer=None):
        super().__init__()
        self.configer = configer
        self.n_datasets = self.configer.get('n_datasets')
        self.num_prototype = _cfg(configer, 'contrast', 'num_prototype')
        self.temperature = _cfg(configer, 'contrast', 'temperature')
        self.with_mulbn = _cfg(configer, 'contrast', 'with_mulbn')
        self.reweight = _cfg(configer, 'loss', 'reweight')
        self.ignore_index = _cfg(configer, 'loss', 'ignore_index', default=255)
        self.with_unify_label = self.configer.get('loss', 'with_unify_label')
        if self.with_unify_label:
            self.classRemapper = eval(self.configer.get('class_remaper'))(configer=self.configer)
        self.n_cats = [configer.get('dataset' + str(i), 'n_cats') for i in range(1, self.n_datasets + 1)]
        self.CELoss = OhemCELoss(0.7, ignore_lb=255)
        self._graph_cache = ops.BipartiteGraphs()
        self._matrices = None

    def forward(self, preds, target, dataset_ids, is_warmup=False):
        logits = preds['seg']
        text_feature_vecs = preds['prototypes']
        present = _present_rows(dataset_ids, self.n_datasets)
        if self.with_unify_label:
            if self._matrices is None or self._matrices[0].device != logits.device:
                self._matrices = [self.classRemapper.getRemapMatrix(i).to(logits.device)
                                  for i in range(self.n_datasets)]
            graphs = self._matrices
            if FOLD_PROTOTYPES:  # :692 + :701 as one contraction with remap_matrix @ text features
                per_ds = ops.mds_head_proj_ohem_ce(logits, text_feature_vecs[self.n_datasets], target, dataset_ids,
                                                   graphs, float(self.CELoss.thresh), self.CELoss.ignore_lb,
                                                   per_dataset=True)
                return _sum_present(per_ds, present)
            logits = ops.prototype_head(logits, text_feature_vecs[self.n_datasets])  # :692 on tcgen05
        else:
            graphs = [text_feature_vecs[i] for i in range(self.n_datasets)]
        per_ds = ops.mds_proj_ohem_ce(logits, target, dataset_ids, graphs, float(self.CELoss.thresh),
                                      self.CELoss.ignore_lb, cache=self._graph_cache, per_dataset=True)
        return _sum_present(per_ds, present)


class CrossDatasetsCELoss_GNN(nn.Module):
    """:714-776 — prototype head, bipartite projection, bilinear up-sampling, plain cross-entropy per dataset (+ the
    sparsity / max-entropy graph regularisers), summed over the datasets present."""

    def __init__(self, configer=None):
        super().__init__()
        self.configer = configer
        self.n_datasets = self.configer.get('n_datasets')
        self.num_prototype = _cfg(configer, 'contrast', 'num_prototype')
        self.temperature = _cfg(configer, 'contrast', 'temperature')
        self.with_mulbn = _cfg(configer, 'contrast', 'with_mulbn')
        self.reweight = _cfg(configer, 'loss', 'reweight')
        self.ignore_index = _cfg(configer, 'loss', 'ignore_index', default=255)
        self.with_unify_label = _cfg(configer, 'loss', 'with_unify_label')
        self.with_spa = _cfg(configer, 'loss', 'with_spa', default=False)
        self.spa_loss_weight = _cfg(configer, 'loss', 'spa_loss_weight', default=0.0)
        self.with_max_enc = _cfg(configer, 'loss', 'with_max_enc', default=False)
        self.max_enc_weight = _cfg(configer, 'loss', 'max_enc_weight', default=0.0)
        self.n_cats = [configer.get('dataset' + str(i), 'n_cats') for i in range(1, self.n_datasets + 1)]
        self.CELoss = torch.nn.CrossEntropyLoss(ignore_index=255)  # kept for introspection only
        if self.with_max_enc:
            self.MSE_loss = torch.nn.MSELoss()
        self._graph_cache = ops.BipartiteGraphs()

    def forward(self, preds, target, dataset_ids, is_warmup=False):
        logits = preds['seg']
        unify_prototype = preds['unify_prototype']
        bi_graphs = preds['bi_graphs']
        present = _present_rows(dataset_ids, self.n_datasets)
        if FOLD_PROTOTYPES:  # :747 + :759 as one contraction with bi_graph @ unify_prototype
            per_ds = ops.mds_head_proj_ce_mean(logits, unify_prototype, target, dataset_ids,
                                               list(bi_graphs)[:self.n_datasets], ignore=255)
        else:
            logits = ops.prototype_head(logits, unify_prototype)  # :747 on tcgen05
            per_ds = ops.mds_proj_ce_mean(logits, target, dataset_ids, list(bi_graphs)[:self.n_datasets], ignore=255,
                                          cache=self._graph_cache)
        loss = _sum_present(per_ds, present)
        for i in range(self.n_datasets):
            if not present[i]:
                continue
            if self.with_spa:
                loss = loss + self.spa_loss_weight * torch.pow(torch.norm(bi_graphs[i], p='fro'), 2)
            if self.with_max_enc:
                gi = bi_graphs[i]
                loss = loss + self.max_enc_weight * self.MSE_loss(torch.max(gi, dim=1)[0],
                                                                  torch.ones(gi.size(0), device=gi.device))
        return loss


class _GridSplitProjection(torch.autograd.Function):
    """``UnifyPrototypeFunction`` (:779-809): einsum forward; in the backward the gradient of every image is masked
    per unified class by the row ``M[dataset]`` before it reaches the features and the prototypes."""

    @staticmethod
    def forward(ctx, x, weight, dataset_ids, M):
        ctx.save_for_backward(x, weight, dataset_ids, M)
        return torch.einsum('bchw,nc->bnhw', x, weight)

    @staticmethod
    def backward(ctx, g):
        x, weight, dataset_ids, M = ctx.saved_tensors
        valid = (dataset_ids >= 0) & (dataset_ids < M.shape[0])
        rows = M[dataset_ids.clamp(0, M.shape[0] - 1).long()]                       # [B, C_uni]
        rows = torch.where(valid[:, None], rows, torch.ones_like(rows))
        g = g * rows[:, :, None, None].to(g.dtype)
        return torch.einsum('bchw,cn->bnhw', g, weight), torch.einsum('bchw,bnhw->cn', g, x), None, None


class CrossDatasetsCELoss_AdvGNN(nn.Module):
    def __init__(self, configer=None):
        super().__init__()
        self.configer = configer
        g = lambda *k, default=None: _cfg(configer, *k, default=default)
        self.n_datasets = configer.get('n_datasets')
        self.temperature = g('contrast', 'temperature', default=0.07)
        self.ignore_index = g('loss', 'ignore_index', default=255)
        self.with_spa = g('loss', 'with_spa', default=False)
        self.spa_loss_weight = g('loss', 'spa_loss_weight', default=0.0)
        self.with_max_enc = g('loss', 'with_max_enc', default=False)
        self.max_enc_weight = g('loss', 'max_enc_weight', default=0.0)
        self.with_datasets_aux = g('loss', 'with_datasets_aux', default=False)
        self.with_softmax_and_max = g('GNN', 'output_softmax_and_max_adj', default=False)
        self.with_orth = g('GNN', 'with_orth', default=False)
        self.with_max_adj = g('GNN', 'output_max_adj', default=False)
        self.mse_or_adv = g('GNN', 'mse_or_adv', default="None")
        self.gnn_iters = g('train', 'gnn_iters', default=1)
        self.seg_iters = g('train', 'seg_iters', default=0)
        self.n_cats = [configer.get('dataset' + str(i), 'n_cats') for i in range(1, self.n_datasets + 1)]
        self.total_cats = sum(self.n_cats)
        self.max_num_unify_class = int(configer.get('GNN', 'unify_ratio') * self.total_cats)
        self.OhemCELoss = OhemCELoss(0.7, ignore_lb=255)
        self.mdsOhemCELoss = MdsOhemCELoss(configer, 0.4, ignore_lb=255)
        self.advloss = nn.BCELoss()
        self.adv_loss_weight = g('loss', 'adv_loss_weight', default=1)
        self.MSE_loss = nn.MSELoss()
        self.MSE_sum_loss = nn.MSELoss(reduction='sum')
        self.orth_weight = g('GNN', 'orth_weight', default=1)
        if self.with_datasets_aux:
            self.aux_weight = configer.get('loss', 'aux_weight')
        self.adj_loss_weight = g('loss', 'adj_loss_weight', default=1)
        self.GridSpilt = g('loss', 'GridSplit', default=False)  # (sic) the reference's attribute name
        if self.GridSpilt:  # :861-871
            cur = 0
            self.M = torch.zeros(self.n_datasets, self.max_num_unify_class)
            for i in range(self.n_datasets):
                n = int(0.5 * self.max_num_unify_class * self.n_cats[i] / float(self.total_cats))
                self.M[i, cur:cur + n] = 1
                cur += n
            self.M[:, cur:] = 1
        # one descriptor cache per graph set: the hard and the soft graphs of a dataset alternate in one forward
        self._graph_cache = [ops.BipartiteGraphs(assume_onehot01=ASSUME_ONEHOT01_GRAPHS),
                             ops.BipartiteGraphs(assume_onehot01=ASSUME_ONEHOT01_GRAPHS)]

    def similarity_dsb(self, proto_vecs, reduce='mean'):
        """:874-893 — entropy of the soft-max over prototype-prototype dot products."""
        z = torch.mm(proto_vecs, proto_vecs.t()) / self.temperature
        ent = F.softmax(z, dim=1) * F.log_softmax(z, dim=1)
        return -1 * (torch.mean(ent) if reduce == 'mean' else torch.sum(ent))

    # -- helpers ----------------------------------------------------------------------------------------------
    def _present(self, dataset_ids):
        return _present_rows(dataset_ids, self.n_datasets)

    def _fused_ce(self, logits, target, dataset_ids, graphs, which, head=None):
        if head is not None:  # `logits` are the features: einsum :971 and einsum :996-1006 folded into one contraction
            return ops.mds_head_proj_ohem_ce(logits, head, target, dataset_ids, list(graphs),
                                             float(self.mdsOhemCELoss.thresh), self.mdsOhemCELoss.ignore_lb)
        return ops.mds_proj_ohem_ce(logits, target, dataset_ids, list(graphs), float(self.mdsOhemCELoss.thresh),
                                    self.mdsOhemCELoss.ignore_lb, cache=self._graph_cache[which])

    def forward(self, preds, target, dataset_ids, is_adv=True, init_gnn_stage=False):
        logits = preds['seg']
        dev = logits.device
        isSecondStage = preds.get('gnn_stage', False)
        unify_prototype = preds.get('unify_prototype')
        bi_graphs = preds['bi_graphs']
        adj_matrix = preds.get('adj')
        target_bi_graph = preds.get('target_bi_graph')
        rows_of = self._present(dataset_ids)
        index_of = [torch.tensor(r, dtype=torch.long, device=dev) if r else None for r in rows_of]
        pairs = len(bi_graphs) == 2 * self.n_datasets

        loss = orth_loss = aux_loss = adj_loss = None
        add = lambda acc, v: v if acc is None else acc + v

        # ---- prototype head (:941-972): tcgen05 GEMMs (ops.prototype_head) ----
        proto_aux = None
        fold_head = None  # set: `logits` stay the features and the loss folds the prototypes into the graphs
        if unify_prototype is not None and not init_gnn_stage:
            feats = logits
            head = unify_prototype
            if self.with_datasets_aux:
                proto_aux, cur = [], 0
                for i in range(self.n_datasets):
                    if index_of[i] is None:
                        proto_aux.append(None)
                    else:  # low resolution; the up-sampling is fused into the loss kernel below
                        proto_aux.append(ops.prototype_head(feats.index_select(0, index_of[i]),
                                                            unify_prototype[cur:cur + self.n_cats[i]]))
                    cur += self.n_cats[i]
                head = unify_prototype[self.total_cats:]
            if self.GridSpilt:
                self.M = self.M.to(dev)
                logits = _GridSplitProjection.apply(feats, head, torch.as_tensor(dataset_ids).to(dev), self.M)
            elif FOLD_PROTOTYPES:
                fold_head = head
            else:
                logits = ops.prototype_head(feats, head)

        if is_adv and self.with_orth:  # :977-982
            orth_loss = self.orth_weight * self.similarity_dsb(
                unify_prototype[self.total_cats:] if self.with_datasets_aux else unify_prototype)

        blend = (not init_gnn_stage) and is_adv and self.with_softmax_and_max and self.with_max_adj and pairs
        if not init_gnn_stage and is_adv and self.with_softmax_and_max and self.with_max_adj and pairs and isSecondStage:
            # :996 builds bi_graphs[i]-projected logits in the second stage but :1063 still blends the (empty) pair
            # lists; MdsOhemCELoss then fails on the list lengths.  Surface that instead of guessing.
            raise RuntimeError("gnn_stage=True with 2*n_datasets graphs: the reference fails in MdsOhemCELoss here")

        # ---- per-dataset graph regularisers and aux heads (:989-1056), present datasets only ----
        aux_terms = []
        for i in range(self.n_datasets):
            if index_of[i] is None:
                continue
            if is_adv and self.with_spa and not isSecondStage and pairs:  # :1013-1021
                loss = add(loss, self.spa_loss_weight * torch.pow(torch.norm(bi_graphs[2 * i + 1], p='fro'), 2))
            if is_adv and self.with_max_enc:  # :1023-1028
                gi = bi_graphs[i]
                loss = add(loss, self.max_enc_weight * self.MSE_loss(torch.max(gi, dim=1)[0],
                                                                      torch.ones(gi.size(0), device=gi.device)))
            if is_adv and target_bi_graph is not None and not isSecondStage:  # :1030-1043
                gi = bi_graphs[2 * i + 1] if pairs else bi_graphs[i]
                keep = target_bi_graph[i] != 255
                adj_loss = add(adj_loss, (1 / bi_graphs[i].shape[1]) * self.MSE_sum_loss(gi[keep], target_bi_graph[i][keep]))
            if self.with_datasets_aux:
                if is_adv:  # :1045-1049 — heads from the dataset prototypes
                    if proto_aux is None:
                        raise RuntimeError("with_datasets_aux in the GNN stage needs preds['unify_prototype']")
                    aux_terms.append(ops.up_ohem_ce([proto_aux[i]], target.index_select(0, index_of[i]), None,
                                                    float(self.OhemCELoss.thresh), self.OhemCELoss.ignore_lb,
                                                    seg_per_dataset=False)[0])
        if self.with_datasets_aux and not is_adv:  # :1050-1056 — heads from the net, all datasets in one launch set
            per_ds = ops.up_ohem_ce(list(preds['aux']), target, dataset_ids, float(self.OhemCELoss.thresh),
                                    self.OhemCELoss.ignore_lb, seg_per_dataset=True)
            aux_terms = [per_ds[i] for i in range(self.n_datasets) if index_of[i] is not None]
        for t in aux_terms:
            aux_loss = add(aux_loss, t)

        # ---- the segmentation loss (:1062-1080) ----
        if not init_gnn_stage:
            if blend:
                cur_iter = self.configer.get('iter')
                cur_iter = cur_iter % (self.gnn_iters + self.seg_iters) % self.gnn_iters
                max_rate = float(cur_iter) / self.gnn_iters
                if fold_head is not None:  # hard and soft losses from one pass over the features per direction
                    pair = ops.mds_head_proj_ohem_ce_heads(logits, fold_head, target, dataset_ids,
                                                           [bi_graphs[0::2], bi_graphs[1::2]],
                                                           float(self.mdsOhemCELoss.thresh), self.mdsOhemCELoss.ignore_lb)
                    ce = max_rate * pair[0] + (1 - max_rate) * pair[1]
                else:
                    ce = (max_rate * self._fused_ce(logits, target, dataset_ids, bi_graphs[0::2], 0)
                          + (1 - max_rate) * self._fused_ce(logits, target, dataset_ids, bi_graphs[1::2], 1))
                loss = add(loss, ce)
            else:
                if pairs:
                    raise RuntimeError("2*n_datasets graphs outside the soft/max GNN stage: the reference indexes "
                                       "bi_graphs[i] (:1006) and mixes hard and soft graphs of different datasets")
                ce = self._fused_ce(logits, target, dataset_ids, bi_graphs, 0, fold_head)
                loss = ce if loss is None else torch.where(torch.isnan(loss), ce, loss + ce)  # :1076-1079

        if init_gnn_stage and adj_matrix is not None:  # :1090-1106
            pretrain = preds['pretrain_bipart_graph']
            graph_loss, cur = None, 0
            for j in range(self.n_datasets):
                cur += self.n_cats[j]
                graph_loss = add(graph_loss, 10 * self.MSE_loss(adj_matrix[cur - self.n_cats[j]:cur, self.total_cats:],
                                                                pretrain[j]))
            loss = add(loss, graph_loss)
        if init_gnn_stage:  # :1108-1113
            loss = add(loss, self.n_datasets * 10 * self.MSE_loss(unify_prototype, logits))

        if is_adv and self.mse_or_adv != "None":  # :1115-1126
            adv_out = preds['adv_out']
            heads = ('ADV1', 'ADV2', 'ADV3')
            if self.mse_or_adv == 'adv':
                real = torch.zeros(adv_out['ADV1'][0].shape[0], 1, device=adv_out['ADV1'][0].device)
                loss = loss + self.adv_loss_weight * sum(self.advloss(adv_out[k][2], real) for k in heads)
            elif self.mse_or_adv == 'mse':
                loss = loss + self.adv_loss_weight * sum(self.MSE_loss(adv_out[k][1], adv_out[k][0]) for k in heads)

        if aux_loss is not None:
            loss = loss + self.aux_weight * aux_loss
        if orth_loss is not None:
            loss = loss + orth_loss
        if adj_loss is not None:
            loss = loss + self.adj_loss_weight * adj_loss
        return loss, orth_loss, aux_loss, adj_loss


UnifyPrototypeFunction = _GridSplitProjection  # the reference's name (:779)

_NATIVE = ("CrossDatasetsCELoss", "CrossDatasetsCELoss_CLIP", "CrossDatasetsCELoss_GNN", "CrossDatasetsCELoss_AdvGNN",
           "LabelToOneHot", "UnifyPrototypeFunction", "OhemCELoss", "MdsOhemCELoss", "MdsOhemNLLPlusLoss", "ClassRemap",
           "ClassRemapOneHotLabel")
__getattr__ = _reference.module_getattr("lib.loss.loss_cross_datasets", _NATIVE)
