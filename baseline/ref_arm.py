"""Reference arm of bench.py: the UNMODIFIED reference modules (learning/*, compiled to oracle/_ref/ by
oracle/build_ref.py) driven through their own public API on the host CPU —
pointnet.PointNet / CloudEmbedder.run, graphnet.GraphNetwork (use_pyg=0, cuda=False: the
reference's own CPU code path incl. the per-node loops of ecc/GraphConvModule.py:82-88,114-121),
ecc.GraphConvInfo, cross entropy, element-wise clamp, torch.optim.Adam (learning/main.py:199-213;
eval: main.py:229-264).  None of this repository's kernels, modules or oracle is on this path.

`igraph` is absent from the image and is only touched by GraphConvInfo.set_batch; the batch's
(idxn, degrees, edge features) — what set_batch would have produced — are handed to the reference's
GraphConvInfo object directly.
"""
import os
import sys
import types
from types import SimpleNamespace

import torch

from oracle import build_ref

REF = build_ref.DST


def available():
    return build_ref.available()


def _import():
    sys.modules.setdefault("igraph", types.ModuleType("igraph"))
    for p in (os.path.join(REF, "learning"), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from learning import ecc, graphnet, pointnet  # noqa: E402  (the reference's own packages)
    return ecc, graphnet, pointnet


class ReferenceStep(object):
    """One reference model + optimizer; `.train_step(batch)` / `.eval_step(batch)` on CPU tensors."""

    def __init__(self, margs, seed=1):
        ecc, graphnet, pointnet = _import()
        self.ecc = ecc
        torch.manual_seed(seed)
        model = torch.nn.Module()
        nfeat = margs.ptn_widths[1][-1]
        # learning/main.py:414-431 (create_model)
        model.ecc = graphnet.GraphNetwork(margs.model_config, nfeat, [margs.edge_feats] + margs.fnet_widths,
                                          margs.fnet_orthoinit, margs.fnet_llbias, margs.fnet_bnidx,
                                          margs.edge_mem_limit, use_pyg=0, cuda=False)
        model.ptn = pointnet.PointNet(margs.ptn_widths[0], margs.ptn_widths[1], margs.ptn_widths_stn[0],
                                      margs.ptn_widths_stn[1], margs.node_feats, margs.ptn_nfeat_stn,
                                      prelast_do=margs.ptn_prelast_do)
        self.model, self.margs = model, margs
        self.embedder = pointnet.CloudEmbedder(SimpleNamespace(cuda=False, ptn_mem_monger=margs.ptn_mem_monger))
        self.opt = torch.optim.Adam(model.parameters(), lr=margs.lr, weight_decay=margs.wd)

    def load(self, sd_ecc, sd_ptn):
        self.model.ecc.load_state_dict(sd_ecc)
        self.model.ptn.load_state_dict(sd_ptn)

    def _info(self, batch):
        gi = self.ecc.GraphConvInfo()
        gi._idxn, gi._idxe = batch["idxn"], None
        gi._degrees, gi._degrees_gpu = batch["degs"], None
        gi._edgefeats = batch["edgefeats"]
        # [2,E] (source, target) pairs as set_batch builds them (GraphConvInfo.py:58,69); only read by
        # the PyG branch, which use_pyg=0 never takes
        tgt = torch.repeat_interleave(torch.arange(batch["degs"].numel()), batch["degs"])
        gi._edge_indexes = torch.stack([batch["idxn"], tgt])
        return gi

    def train_step(self, batch):
        """main.py:199-213."""
        m = self.model
        m.train()
        m.ecc.set_info([self._info(batch)], False)
        self.opt.zero_grad()
        emb = self.embedder.run(m, None, batch["clouds_flag"], batch["clouds"], batch["clouds_global"])
        out = m.ecc(emb)
        loss = torch.nn.functional.cross_entropy(out, batch["labels"])
        loss.backward()
        self.embedder.bw_hook()
        if self.margs.grad_clip > 0:
            for p in m.parameters():
                p.grad.data.clamp_(-self.margs.grad_clip, self.margs.grad_clip)
        self.opt.step()
        return float(loss.detach()), out.detach()

    @torch.no_grad()
    def eval_step(self, batch):
        """main.py:229-264."""
        m = self.model
        m.eval()
        m.ecc.set_info([self._info(batch)], False)
        emb = self.embedder.run(m, None, batch["clouds_flag"], batch["clouds"], batch["clouds_global"])
        return m.ecc(emb)
