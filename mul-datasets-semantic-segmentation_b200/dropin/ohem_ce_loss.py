"""Drop-in for lib/loss/ohem_ce_loss.py (OhemCELoss :12-34, MdsOhemCELoss :36-90, MdsOhemNLLPlusLoss :92-146).

Same constructors, same ``forward`` signatures, same attributes (`thresh` as a 0-dim fp32 tensor holding
-log(p), `ignore_lb`); the arithmetic runs in libmdseg_b200.so.  Differences a caller can observe:
  * no host synchronisation in OhemCELoss.forward (the reference syncs twice through ``.numel()``);
    the result is a 0-dim CUDA tensor, NaN when no pixel is selected (``torch.mean`` of an empty tensor);
  * labels outside [0, C) other than `ignore_lb` do not trip a device assert: they raise a RuntimeError at
    the next ``mdseg_b200.ops.check_errors()``.
"""
import torch
import torch.nn as nn

from .. import ops
from . import _reference


class OhemCELoss(nn.Module):
    def __init__(self, thresh, ignore_lb=255):
        super().__init__()
        self.thresh = -torch.log(torch.tensor(thresh, requires_grad=False, dtype=torch.float))
        self.ignore_lb = ignore_lb
        self.criteria = nn.CrossEntropyLoss(ignore_index=ignore_lb, reduction='none')  # kept for introspection only

    def forward(self, logits, labels):
        """logits [N, C, H, W] (fp32 / fp16 / bf16, NCHW or channels_last), labels [N, H, W] -> 0-dim fp32."""
        return ops.ohem_ce(logits, labels, float(self.thresh), self.ignore_lb)

    def forward_fused(self, logits_lowres, labels):
        """forward(F.interpolate(logits_lowres, size=labels.shape[-2:], mode='bilinear', align_corners=False), labels)
        without the up-sampled tensor: a BiSeNet SegmentHead's trailing nn.Upsample fused into the loss, forward and
        backward.  logits_lowres [N, C, h, w] (NCHW or channels_last), H = f h and W = f w with f in {2, 4, 8, 16}
        per axis; other shapes raise ValueError."""
        return ops.up_ohem_ce([logits_lowres], labels, None, float(self.thresh), self.ignore_lb,
                              align_corners=False)[0]


class MdsOhemCELoss(nn.Module):
    def __init__(self, configer, thresh, ignore_lb=255):
        super().__init__()
        self.configer = configer
        self.n_datasets = self.configer.get('n_datasets')
        self.thresh = -torch.log(torch.tensor(thresh, requires_grad=False, dtype=torch.float))
        self.ignore_lb = ignore_lb
        self.criteria = nn.CrossEntropyLoss(ignore_index=ignore_lb, reduction='none')

    def forward(self, logits, labels, dataset_ids):
        """Reference call form (loss_cross_datasets.py:1074): `logits` is the list of already up-sampled
        per-dataset logits [B_k, C_k, H, W] of the datasets PRESENT in the batch, in ascending dataset id.
        Finding which datasets are present needs the ids on the host (the reference's `.any()` does the same);
        use `forward_fused` to stay on the device."""
        ids = torch.as_tensor(dataset_ids)
        present = sorted(set(int(v) for v in ids.tolist()) & set(range(self.n_datasets)))
        if len(present) != len(logits):
            raise ValueError(f"{len(logits)} logit tensors for {len(present)} datasets present in the batch")
        ids = ids.to(labels.device)
        lbs = [labels[ids == i] for i in present]
        return ops.mds_ohem_ce_full(list(logits), lbs, float(self.thresh), self.ignore_lb)

    def forward_fused(self, logits_uni, labels, dataset_ids, bi_graphs):
        """Projection + bilinear up-sampling + CE + one OHEM selection from the LOW-resolution unified logits
        [B, C_uni, h, w] (loss_cross_datasets.py:1006-1007 + :1074 in one autograd node; no host sync once the graphs' descriptors are
        cached, see ops.mds_proj_ohem_ce).  channels_last logits with 0/1 graphs are taken as they are (no layout copy)
        and get a channels_last gradient."""
        return ops.mds_proj_ohem_ce(logits_uni, labels, dataset_ids, list(bi_graphs), float(self.thresh),
                                    self.ignore_lb)


class MdsOhemNLLPlusLoss(nn.Module):
    """lib/loss/ohem_ce_loss.py:92-146 — the "softmax in the unified space, project PROBABILITIES, up-sample, -log"
    variant (AdjNLLPlusLoss, lib/loss/loss_helper.py:647-668) under one OHEM selection over the batch.

    forward(logits [B, C_uni, h, w], labels [B, H, W], bi_graphs (list of [C_ds_i, C_uni]), dataset_ids [B]).
    The reference's loss vector holds the valid pixels only; here ignored pixels stay in with loss 0, which changes
    neither the threshold set nor the top-n_min set (n_min = #valid // 16).  Unlike the reference, the labels are
    not modified in place (loss_helper.py:662 writes 0 into a COPY made by boolean indexing there as well)."""

    def __init__(self, configer, thresh, ignore_lb=255):
        super().__init__()
        self.configer = configer
        self.n_datasets = self.configer.get('n_datasets')
        self.thresh = -torch.log(torch.tensor(thresh, requires_grad=False, dtype=torch.float))
        self.ignore_lb = ignore_lb
        self._graph_cache = ops.BipartiteGraphs()

    def forward(self, logits, labels, bi_graphs, dataset_ids):
        graphs = list(bi_graphs)[:self.n_datasets]
        return ops.mds_nll_plus(logits, labels, dataset_ids, graphs, float(self.thresh), self.ignore_lb,
                                cache=self._graph_cache)


# RecallCrossEntropy / FocalLoss / AdjNLLPlusLoss (re-exported by the reference module, :10) and anything else:
# the reference's own definitions
__getattr__ = _reference.module_getattr("lib.loss.ohem_ce_loss", ("OhemCELoss", "MdsOhemCELoss", "MdsOhemNLLPlusLoss"))
