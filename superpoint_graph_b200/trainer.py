"""The training / inference step of the reference's trainer on the sm_100a path.

What `learning/main.py:189-221` does per batch — set_info, zero_grad, PointNet embedding, graph
network, weighted cross entropy, backward, element-wise gradient clamp, Adam, logits to the host —
with the model's parameters living in ONE flat fp32 buffer so that the gradient all-reduce is a
single NCCL call and clamp+Adam a single kernel (scene-parallel data parallelism: every rank
owns whole scenes, the graph never crosses devices).
"""
import copy
from types import SimpleNamespace

import torch
import torch.nn as nn

from . import ops
from .spg_ecc import GraphConvInfo
from .spg_graphnet import GraphNetwork
from .spg_pointnet import CloudEmbedder, PointNet, prepack_weights

S3DIS_ARGS = dict(
    model_config="gru_10_1_1_1_0,f_13", ptn_widths=[[64, 64, 128, 128, 256], [256, 64, 32]],
    ptn_widths_stn=[[64, 64, 128], [128, 64]], ptn_nfeat_stn=14, ptn_prelast_do=0,
    ptn_mem_monger=0, fnet_widths=[32, 128, 64], fnet_llbias=0, fnet_orthoinit=1, fnet_bnidx=2,
    edge_mem_limit=30000, node_feats=14, edge_feats=13, classes=13, lr=1e-2, grad_clip=1.0,
    wd=0.0, cuda=1, use_pyg=0)


def make_args(**overrides):
    d = dict(S3DIS_ARGS)
    d.update(overrides)
    return SimpleNamespace(**d)


def create_model(args):
    """ref: learning/main.py:414-431 (`model.ecc` is registered before `model.ptn`)."""
    model = nn.Module()
    nfeat = args.ptn_widths[1][-1]
    model.ecc = GraphNetwork(args.model_config, nfeat, [args.edge_feats] + args.fnet_widths,
                             args.fnet_orthoinit, args.fnet_llbias, args.fnet_bnidx,
                             args.edge_mem_limit, use_pyg=args.use_pyg, cuda=args.cuda)
    model.ptn = PointNet(args.ptn_widths[0], args.ptn_widths[1], args.ptn_widths_stn[0],
                         args.ptn_widths_stn[1], args.node_feats, args.ptn_nfeat_stn,
                         prelast_do=args.ptn_prelast_do)
    return model


def flatten_parameters(model):
    """Moves every parameter into one contiguous fp32 buffer (parameters become views)."""
    params = [p for p in model.parameters()]
    total = sum(p.numel() for p in params)
    flat = torch.empty(total, dtype=torch.float32, device=params[0].device)
    off = 0
    for p in params:
        n = p.numel()
        flat[off:off + n].copy_(p.data.reshape(-1))
        p.data = flat[off:off + n].view(p.shape)
        off += n
    return flat, params


class HostBatch(object):
    """One collated batch in pinned host memory, in the layout the reference's collate produces
    (learning/spg.py:178-193): clouds, global features, edge features, labels and the (idxn, degs) pair of
    GraphConvInfo.set_batch.  The CSR views the kernels read are built ON THE DEVICE from that pair on every
    upload (ops.graph_build_into -> spg_graph_build), inside the timed end-to-end region."""

    FIELDS = ("clouds", "clouds_global", "edgefeats", "labels", "idx_valid", "idxn", "degs")

    def __init__(self, batch):
        self.n_nodes = int(batch["degs"].numel())
        flag = batch["clouds_flag"]
        self.idx_valid = torch.nonzero(flag.eq(0)).reshape(-1)
        self.clouds = batch["clouds"]
        self.clouds_global = batch["clouds_global"]
        self.edgefeats = batch["edgefeats"]
        self.labels = batch["labels"]
        self.idxn = torch.as_tensor(batch["idxn"], dtype=torch.long).contiguous()
        self.degs = torch.as_tensor(batch["degs"], dtype=torch.long).contiguous()
        # the checks of the host builder (ops.EccGraph.__init__), once per batch on the host arrays: the
        # device builder then runs without reading its status word back
        if int(self.degs.sum()) != self.idxn.numel() or (self.degs.numel() and int(self.degs.min()) < 0):
            raise ValueError("sum(degs)=%d does not match the number of edges %d"
                             % (int(self.degs.sum()), self.idxn.numel()))
        if self.idxn.numel() and (int(self.idxn.min()) < 0 or int(self.idxn.max()) >= self.n_nodes):
            raise ValueError("idxn out of range")
        self.gi = GraphConvInfo.from_arrays(self.idxn, self.degs, self.edgefeats)
        if torch.cuda.is_available():
            for f in self.FIELDS:
                setattr(self, f, getattr(self, f).pin_memory())

    def h2d_bytes(self):
        return int(sum(getattr(self, f).numel() * getattr(self, f).element_size() for f in self.FIELDS))

    def to_device(self, device, skip=()):
        """Asynchronous copies + the device graph build on the current stream; returns a DeviceBatch.
        Fields named in `skip` stay on the host (Trainer.eval_step_host uploads the clouds itself)."""
        device = torch.device(device)
        d = DeviceBatch()
        for f in self.FIELDS:
            setattr(d, f, getattr(self, f) if f in skip else getattr(self, f).to(device, non_blocking=True))
        g = ops.EccGraph.from_device(d.idxn, d.degs, n_in=self.n_nodes, check=False)
        d.gi = copy.copy(self.gi)  # (shallow: one GraphConvInfo per device batch, sharing the host arrays)
        d.gi._graph = g  # the kernels read the graph through GraphConvInfo.graph().to(device)
        d.gi._edgefeats = d.edgefeats
        d.n_nodes = self.n_nodes
        return d

    def copy_into(self, d):
        """Asynchronous H2D refresh of an existing DeviceBatch of the same shapes (static buffers of a
        captured CUDA graph), and the rebuild of its graph views in place."""
        for f in self.FIELDS:
            getattr(d, f).copy_(getattr(self, f), non_blocking=True)
        dev = d.gi.graph()._dev[(d.clouds.device.type, d.clouds.device.index)]
        ops.graph_build_into(dev, d.idxn, d.degs, self.n_nodes)


class DeviceBatch(object):
    pass


class Trainer(object):
    """zero_grad / forward / loss / backward / (all-reduce) / clamp / Adam, as one object."""

    def __init__(self, model, args, class_weights=None, process_group=None, world_size=1, dtype="f32"):
        if dtype not in ("f32", "bf16"):
            raise ValueError("dtype must be 'f32' or 'bf16'")
        self.model, self.args, self.dtype = model, args, dtype
        self.flat, self.params = flatten_parameters(model)
        self.flat_grad = torch.zeros_like(self.flat)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_count = 0
        self._generation = 0  # bumped whenever the parameters change (see _params_changed)
        self._learned_packs = {}  # weight images packed on demand by earlier steps (see compute_gradients)
        self._side = ops.SideStream(self.flat.device) if (self.flat.is_cuda and ops.USE_SIDE_STREAM[0]) else None
        self._capturing = False
        self.side_in_eager = False  # tests: exercise the two-stream schedule without a graph
        self.step_dev = torch.zeros((), dtype=torch.int64, device=self.flat.device)
        self._graphs = {}
        self.class_weights = class_weights
        self.pg, self.world_size = process_group, world_size
        self._fused_ar = None
        if world_size > 1:  # one-time setup collective: guarantee identical replicas
            torch.distributed.broadcast(self.flat, 0, group=process_group)
            if self.flat.is_cuda and ops.USE_FUSED_ALLREDUCE[0]:
                # gradient buffer in symmetric memory: all-reduce + clamp + Adam become ONE kernel over
                # NVLink peer pointers; any failure to set that up leaves the NCCL path in place
                try:
                    self._fused_ar = ops.FusedAllreduce(self.flat.numel(), self.flat.device,
                                                        process_group or torch.distributed.group.WORLD)
                    self.flat_grad = self._fused_ar.grad
                except Exception as ex:  # pragma: no cover (depends on the box's P2P capabilities)
                    import warnings
                    warnings.warn("fused all-reduce unavailable (%r): using torch.distributed.all_reduce" % (ex,))
                    self._fused_ar = None
        self.embedder = CloudEmbedder(SimpleNamespace(cuda=1, ptn_mem_monger=args.ptn_mem_monger))

    def forward(self, db):
        for gc in self.model.ecc.gconvs:  # one batched graph, shared by every convolution of the model
            gc.set_info(db.gi)
        if ops.SIDE[0] is not None:  # filter networks run underneath the PointNet forward
            for gc in self.model.ecc.gconvs:
                if hasattr(gc, "prefetch_filters"):
                    gc.prefetch_filters()
        # CloudEmbedder.run's device-resident twin (same code path behind it, incl. mem-monger)
        emb = self.embedder.run_resident(self.model, db.clouds, db.clouds_global, db.idx_valid, db.n_nodes)
        return self.model.ecc(emb)

    def compute_gradients(self, db):
        """Forward, loss, backward; gathers every parameter gradient into the flat buffer.
        Returns (loss[1], logits).  Purely local to this rank (no collective)."""
        # launch policy (ops.set_pdl): programmatic dependent launch measured 2 % SLOWER on the training step —
        # for the whole step and for the forward phase alone (profiles/r2_pdl_policy_ab.log) — so it is off
        # here; the inference paths leave it on
        ops.set_pdl(0)
        try:
            return self._compute_gradients(db)
        finally:
            ops.set_pdl(1)

    def _compute_gradients(self, db):
        if self.dtype != "f32":
            raise NotImplementedError("training runs in fp32 (3xTF32 on the tensor cores); bf16 arithmetic is "
                                      "implemented for the inference forward only (Trainer.eval_step)")
        self.model.train()
        for p in self.params:
            p.grad = None
        # weight images: the point-wise layers are known in advance, the rest (FC layers, filter net,
        # classifier) is learned from the on-demand packs of the previous step -> one launch
        self._prepack(db)
        ops.PACK_LEARN[0] = self._learned_packs
        # the second stream pays off where the GPU is the bottleneck (graph replay); eager steps are
        # bound by the CPU issuing ~250 launches, and every fork costs host time
        use_side = self._side is not None and (self._capturing or self.side_in_eager)
        ops.SIDE[0] = self._side if use_side else None
        try:
            logits = self.forward(db)
            loss, d_logits = ops.ce_loss(logits, db.labels, self.class_weights, -100)
            logits.backward(d_logits)
            self.embedder.bw_hook()
        finally:
            ops.PACK_LEARN[0] = None
            ops.SIDE[0] = None
            if use_side:
                self._side.join()
        ops.PACK_CACHE.clear()  # the optimizer is about to change the weights
        torch.cat([p.grad.reshape(-1) for p in self.params], out=self.flat_grad)
        return loss, logits.detach()

    def _prepack(self, db):
        prepack_weights(self.model.ptn, db.clouds.shape[0], db.clouds.shape[2],
                        extra=list(self._learned_packs.values()))

    def apply_update(self):
        """One all-reduce of the flat gradient (scene-parallel ranks), then clamp + Adam in one
        kernel (gradient averaged by 1/world before the clamp, as main.py:210-213 on one GPU)."""
        self.step_count += 1
        if self._fused_ar is not None:
            self._fused_ar.step_(self.flat, self.exp_avg, self.exp_avg_sq, self.step_dev, lr=self.args.lr,
                                 weight_decay=self.args.wd, grad_clip=self.args.grad_clip)
        else:
            self.reduce_gradients()
            ops.clamp_adam_dev_(self.flat, self.flat_grad, self.exp_avg, self.exp_avg_sq, self.step_dev,
                                lr=self.args.lr, weight_decay=self.args.wd, grad_clip=self.args.grad_clip,
                                grad_scale=1.0 / self.world_size)
        self._params_changed()

    def _params_changed(self):
        """The parameters were written through `flat`, behind torch's back.  Bump their version counters,
        one per tensor (the parameters are views of `flat` with counters of their own): caches keyed on
        versions (the folded eval weight images) then rebuild, and eval graphs captured before this point
        refuse to replay."""
        torch.autograd.graph.increment_version(self.params)
        self._generation += 1

    def reduce_gradients(self):
        """The step's only collective: SUM of the flat gradient over the scene-parallel ranks (the
        1/world average is applied inside the clamp+Adam kernel, before the clamp)."""
        if self.world_size > 1:
            torch.distributed.all_reduce(self.flat_grad, group=self.pg)
        return self.flat_grad

    def train_step(self, db):
        """One optimisation step on a device-resident batch; returns (loss[1], logits)."""
        loss, logits = self.compute_gradients(db)
        self.apply_update()
        return loss, logits

    # ---- CUDA-graph replay for batches whose shapes repeat (fixed-size evaluation resampling,
    # synthetic sweeps).  The local part of the step (forward, loss, backward, gradient gather) is
    # static given the shapes: one capture, then one graph launch per step instead of ~250 kernel
    # launches.  The collective and the optimizer kernel stay outside the graph (NCCL is not
    # captured).  Batches of new shapes simply run eagerly.
    def _snapshot(self):
        bufs = [b for b in self.model.buffers()]
        return (self.flat.clone(), self.exp_avg.clone(), self.exp_avg_sq.clone(), self.step_dev.clone(),
                self.step_count, bufs, [b.clone() for b in bufs])

    def _restore(self, snap):
        flat, m, v, step_dev, step_count, bufs, saved = snap
        self.flat.copy_(flat)
        self.exp_avg.copy_(m)
        self.exp_avg_sq.copy_(v)
        self.step_dev.copy_(step_dev)
        self.step_count = step_count
        for b, sv in zip(bufs, saved):
            b.copy_(sv)
        self._params_changed()

    def capture(self, db, key=None, warmup=2):
        """Captures compute_gradients on the static tensors of `db`; returns the key for replay().
        Free of side effects: the `warmup` (>= 1) eager steps that prime workspaces, weight-image
        tables and lazy handles run on a snapshot — parameters, Adam state, step count and BatchNorm
        buffers are restored before the capture."""
        if warmup < 1:
            raise ValueError("capture() needs at least one warm-up step (the batched weight packing uploads "
                             "its job table on first use, which cannot happen inside a capture)")
        key = key if key is not None else id(db)
        snap = self._snapshot()
        for _ in range(warmup):
            self.train_step(db)
        self._restore(snap)
        # the job table of the batched weight packing is uploaded on first use: do that outside
        # the capture (a pageable H2D copy cannot be captured)
        self._prepack(db)
        ops.PACK_CACHE.clear()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        self._capturing = True
        try:
            with torch.cuda.graph(g):
                loss, logits = self.compute_gradients(db)
        finally:
            self._capturing = False
        self._graphs[key] = (g, db, loss, logits)
        return key

    def replay(self, key):
        g, db, loss, logits = self._graphs[key]
        g.replay()
        # the replayed forward updated the BatchNorm running statistics without running chain_forward's host code
        torch.autograd.graph.increment_version(list(self.model.buffers()))
        self.apply_update()  # (NCCL path: outside the graph; fused path: one more kernel launch)
        return loss, logits

    @torch.no_grad()
    def eval_step(self, db):
        """Inference forward (main.py:229-264).  dtype "bf16": the PointNet trunk (the tensor-core part of
        the step) runs in bf16 arithmetic with fp32 accumulation; everything behind the pooled rows stays
        fp32."""
        self.model.eval()
        ops.EVAL_BF16[0] = self.dtype == "bf16"
        try:
            return self.forward(db)
        finally:
            ops.EVAL_BF16[0] = False

    def capture_eval(self, db, key=None, warmup=2):
        """Captures the inference forward on the static tensors of `db` (no side effects to undo: eval mode
        updates nothing); returns the key for replay_eval().  One graph launch instead of ~100 kernel
        launches — at a few thousand superpoints the eager forward is issue-bound on the host."""
        key = ("eval", key if key is not None else id(db))
        for _ in range(max(1, warmup)):  # primes workspaces, folded weight images, lazy handles
            self.eval_step(db)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        self._capturing = True
        try:
            with torch.cuda.graph(g):
                logits = self.eval_step(db)
        finally:
            self._capturing = False
        self._graphs[key] = (g, db, self._generation, logits)
        return key

    def replay_eval(self, key):
        """Replays a capture_eval graph.  The graph holds the folded weight images of the parameters it was
        captured with, so it refuses to run once an update changed them: capture again."""
        g, db, generation, logits = self._graphs[key]
        if generation != self._generation:
            raise RuntimeError("replay_eval: the parameters changed since capture_eval (the graph would run the "
                               "old weights); capture the inference forward again")
        g.replay()
        return logits

    @torch.no_grad()
    def eval_step_host(self, hb):
        """Inference straight from a pinned HostBatch: the small arrays go up first, the graph views are built
        on the device, the point clouds follow in chunks on a copy stream while the filter networks and the
        PointNet of the chunks already there run (CloudEmbedder.run_pipelined).  Same result as
        eval_step(hb.to_device(dev)) up to the per-row summation order of the FC layers."""
        self.model.eval()
        ops.EVAL_BF16[0] = self.dtype == "bf16"
        try:
            dev = self.flat.device
            if hb.clouds.numel() * hb.clouds.element_size() < CloudEmbedder.PIPELINE_MIN_BYTES:
                return self.forward(hb.to_device(dev))
            d = hb.to_device(dev, skip=("clouds", "clouds_global"))
            for gc in self.model.ecc.gconvs:
                gc.set_info(d.gi)

            def filters():
                for gc in self.model.ecc.gconvs:
                    if hasattr(gc, "prefetch_filters"):
                        gc.prefetch_filters(inline=True)

            emb = self.embedder.run_pipelined(self.model, hb.clouds, hb.clouds_global, d.idx_valid, d.n_nodes,
                                              overlap=filters)
            return self.model.ecc(emb)
        finally:
            ops.EVAL_BF16[0] = False

    # ---- optimizer state in torch.optim.Adam's layout (checkpoints of main.py:342-346,390-412)
    def optimizer_state_dict(self):
        """{'state': {i: {'step', 'exp_avg', 'exp_avg_sq'}}, 'param_groups': [...]} with one entry per
        parameter in model.parameters() order — what torch.optim.Adam(model.parameters()).state_dict()
        holds after the same number of steps."""
        state, off = {}, 0
        step = int(self.step_dev.item())
        for i, p in enumerate(self.params):
            n = p.numel()
            if step > 0:
                state[i] = {"step": torch.tensor(float(step)),
                            "exp_avg": self.exp_avg[off:off + n].view(p.shape).clone(),
                            "exp_avg_sq": self.exp_avg_sq[off:off + n].view(p.shape).clone()}
            off += n
        group = {"lr": self.args.lr, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": self.args.wd,
                 "amsgrad": False, "maximize": False, "foreach": None, "capturable": False,
                 "differentiable": False, "fused": None, "params": list(range(len(self.params)))}
        return {"state": state, "param_groups": [group]}

    def load_optimizer_state_dict(self, sd):
        off, step = 0, 0
        for i, p in enumerate(self.params):
            n = p.numel()
            st = sd["state"].get(i)
            if st is None:
                self.exp_avg[off:off + n].zero_()
                self.exp_avg_sq[off:off + n].zero_()
            else:
                self.exp_avg[off:off + n].copy_(st["exp_avg"].reshape(-1))
                self.exp_avg_sq[off:off + n].copy_(st["exp_avg_sq"].reshape(-1))
                step = max(step, int(float(st["step"])))
            off += n
        if sd.get("param_groups"):
            self.args.lr = sd["param_groups"][0].get("lr", self.args.lr)
        self.step_dev.fill_(step)
        self.step_count = step


