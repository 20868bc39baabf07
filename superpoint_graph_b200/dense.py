"""Chains of (Linear | Conv1d k=1) [+ BatchNorm1d] [+ ReLU] layers with hand-written forward AND
backward over the C-ABI kernels.

Only the raw (pre-norm) output of each layer is stored; "BatchNorm apply + ReLU" of a layer is
deferred and fused into whatever consumes it (the next layer's GEMM operand load, the
segmented max-pool, or an explicit materialisation at the end of a chain).

Reference semantics: the nn.Sequential stacks built by learning/pointnet.py:27-53,83-118 and
learning/graphnet.py:17-34 (`create_fnet`), in training mode (batch statistics, running-stat
update with momentum, biased variance for normalisation / unbiased for the running estimate) and
in eval mode (running statistics).
"""
import torch
import torch.nn as nn

from . import ops


class LayerSpec(object):
    """One parametric layer: names index into the flat parameter list given to the chain."""

    __slots__ = ("w", "b", "gamma", "beta", "bn", "relu", "cin", "cout")

    def __init__(self, w, b, gamma, beta, bn, relu, cin, cout):
        self.w, self.b, self.gamma, self.beta = w, b, gamma, beta
        self.bn, self.relu, self.cin, self.cout = bn, relu, cin, cout


def parse_sequential(seq, training):
    """nn.Sequential -> ([LayerSpec], [parameter tensors]).  LayerSpec.w/b/gamma/beta are
    positions in the returned parameter list; LayerSpec.bn is the BatchNorm module (buffers)."""
    specs, params = [], []
    mods = list(seq.children()) if isinstance(seq, nn.Sequential) else list(seq)
    i = 0
    while i < len(mods):
        m = mods[i]
        if isinstance(m, nn.Conv1d):
            if m.kernel_size != (1,) or m.stride != (1,) or m.padding != (0,) or m.groups != 1:
                raise NotImplementedError("only 1x1 Conv1d layers are on the SPG path")
            cout, cin = m.weight.shape[0], m.weight.shape[1]
        elif isinstance(m, nn.Linear):
            cout, cin = m.weight.shape
        elif isinstance(m, nn.Dropout):
            if training and m.p > 0:
                raise NotImplementedError(
                    "dropout with p>0 in training mode is not implemented by the fused path "
                    "(the reference's documented configs use ptn_prelast_do=0)")
            i += 1
            continue
        else:
            raise NotImplementedError("unsupported module in fused chain: %r" % (m,))
        w = len(params)
        params.append(m.weight)
        b = None
        if m.bias is not None:
            b = len(params)
            params.append(m.bias)
        i += 1
        bn, gamma, beta, relu = None, None, None, False
        if i < len(mods) and isinstance(mods[i], nn.BatchNorm1d):
            bn = mods[i]
            if bn.affine:
                gamma = len(params)
                params.append(bn.weight)
                beta = len(params)
                params.append(bn.bias)
            i += 1
        elif i < len(mods) and isinstance(mods[i], nn.GroupNorm):
            raise NotImplementedError("norm='layer'/'group' PointNets are not on the fused path")
        if i < len(mods) and isinstance(mods[i], nn.ReLU):
            relu = True
            i += 1
        specs.append(LayerSpec(w, b, gamma, beta, bn, relu, cin, cout))
    return specs, params


class Deferred(object):
    """A raw activation [M, C] (leading dimension ld) plus the affine+ReLU still to be applied."""

    __slots__ = ("raw", "ld", "C", "scale", "shift", "relu")

    def __init__(self, raw, ld, C, scale=None, shift=None, relu=False):
        self.raw, self.ld, self.C = raw, ld, C
        self.scale, self.shift, self.relu = scale, shift, relu

    @property
    def pending(self):
        return self.scale is not None or self.shift is not None or self.relu

    def aff(self):
        return (self.scale, self.shift, self.relu) if self.pending else None

    def materialise(self, M):
        if not self.pending and self.ld == self.C:
            return self.raw
        return ops.affine_act(self.raw, self.ld, M, self.C, self.scale, self.shift, self.relu)


_ZEROS = {}


def _zeros(n, device):
    key = (n, device.index)
    z = _ZEROS.get(key)
    if z is None:
        z = torch.zeros(n, dtype=torch.float32, device=device)
        _ZEROS[key] = z
    return z


def _padded_k(cin, ld):
    """cin rounded up to a multiple of 32 if the rows are wide enough to be read that far."""
    kp = (cin + 31) // 32 * 32
    return kp if kp <= ld else cin


def _w2d(w):
    return w.view(w.shape[0], w.shape[1]) if w.dim() == 3 else w


def chain_forward(inp, M, specs, params, training, saved=None):
    """inp: Deferred input.  Returns the Deferred output of the last layer.  If `saved` is a list,
    per-layer records for chain_backward are appended to it."""
    cur = inp
    for sp in specs:
        W = _w2d(params[sp.w])
        bias = params[sp.b] if sp.b is not None else None
        bn = sp.bn
        batch_stats = bn is not None and (training or not bn.track_running_stats)
        fold = None
        if batch_stats:
            # BatchNorm fold (scale/shift, running statistics, num_batches_tracked) rides on the last
            # level of the statistics merge
            rm = rv = nbt = None
            mom = 0.0
            if training and bn.track_running_stats:
                rm, rv, nbt = bn.running_mean, bn.running_var, bn.num_batches_tracked
                if bn.momentum is None:
                    raise NotImplementedError("BatchNorm momentum=None (cumulative average)")
                mom = bn.momentum
            fold = (params[sp.gamma] if sp.gamma is not None else None,
                    params[sp.beta] if sp.beta is not None else None, bn.eps, rm, rv, nbt, mom)
        kpad = _padded_k(sp.cin, cur.ld)
        if ops.tc_supported(M, sp.cout, kpad, cur.ld, sp.cout) and (kpad == sp.cin or not cur.pending):
            # reduction dimension zero-padded to a multiple of 32 (the rows are zero-padded to
            # cur.ld and the weight image gets zeros there)
            res = ops.tc_gemm(cur.raw, cur.ld, W, sp.cin, False, M, sp.cout, kpad, bias=bias,
                              a_aff=cur.aff(), stats=batch_stats, k_valid=sp.cin, fold=fold)
        else:
            res = ops.gemm(cur.raw, cur.ld, True, W, sp.cin, True, M, sp.cout, sp.cin, bias=bias,
                           a_aff=cur.aff(), stats=batch_stats, fold=fold)
        if fold is not None and fold[3] is not None:
            # the kernel updated the running statistics in place: tell torch, so that caches keyed on
            # version counters (ops.pointnet_fused_image) see the change
            torch.autograd.graph.increment_version([fold[3], fold[4], fold[5]])
        mean = var = scale = shift = None
        y = res
        if bn is not None:
            gamma = params[sp.gamma] if sp.gamma is not None else None
            beta = params[sp.beta] if sp.beta is not None else None
            if batch_stats:
                y, mean, var, scale, shift = res  # statistics + fold come out of the GEMM's merge
            else:
                mean, var = bn.running_mean, bn.running_var
                scale, shift = ops.bn_fold(mean, var, gamma, beta, bn.eps)
        nxt = Deferred(y, sp.cout, sp.cout, scale, shift, sp.relu)
        if saved is not None:
            saved.append((cur, nxt, mean, var))
        cur = nxt
    return cur


def _accumulate_grad(prm, g):
    if prm.requires_grad:
        prm.grad = g if prm.grad is None else prm.grad + g


def chain_backward(G, ldg, M, specs, params, saved, need_input_grad, grads, own_g=False, pooled=None):
    """G: gradient w.r.t. the chain's final *activated* output [M, C_last].
    `grads` (list aligned with params) is filled in place.  Returns the gradient w.r.t. the
    chain input's activated value [M, cin_0] (or None).

    Where the data-gradient GEMM of a layer runs on the tcgen05 kernel, the BatchNorm/ReLU backward
    around it is fused into that ONE launch: the prologue turns dL/d(activation) into dL/dY on the
    fly (and stores it once for the weight-gradient kernel), the epilogue reduces the BatchNorm-
    backward sums of the layer below from the tile it has just produced.  The stand-alone
    act_bwd_reduce / act_bwd_apply kernels remain for the small-row chains."""
    red = None  # s1|s2 of the current layer, if the GEMM that produced G already reduced them
    for li in range(len(specs) - 1, -1, -1):
        sp = specs[li]
        cur, nxt, mean, var = saved[li]
        C = sp.cout
        Wp = params[sp.w]
        want_dx = li > 0 or need_input_grad
        fused_pool = (pooled is not None and li == len(specs) - 1 and sp.bn is not None
                      and mean is not None and C % 4 == 0)
        if G is None and not fused_pool:  # generic path: materialise the dense pooled gradient
            gp, ldgp, argmax, Bc, Lc = pooled
            G, ldg, own_g = ops.segmax_bwd(gp, ldgp, argmax, Bc, Lc, C), C, True
        lazy = None  # BatchNorm backward deferred into the data-gradient GEMM's prologue
        dY, ldy = None, C
        if fused_pool:
            # the chain's output went through a max-pool: fused pool-backward + BN/ReLU backward
            gp, ldgp, argmax, Bc, Lc = pooled
            s1, s2, dY = ops.segmax_bn_bwd(gp, ldgp, argmax, nxt.raw, nxt.ld, nxt.scale, nxt.shift,
                                           mean, var, sp.bn.eps, nxt.relu, Bc, Lc, C)
            if sp.gamma is not None:
                grads[sp.gamma] = s2
                grads[sp.beta] = s1
        elif sp.bn is not None:
            eps = sp.bn.eps
            s12 = red if red is not None else ops.act_bwd_reduce(
                G, ldg, nxt.raw, nxt.ld, nxt.scale, nxt.shift, mean, var, eps, nxt.relu, M, C)
            s1, s2 = s12[:C], s12[C:]
            if sp.gamma is not None:
                grads[sp.gamma] = s2
                grads[sp.beta] = s1
            if (ops.USE_FUSED_BNBWD[0] and want_dx and ldg % 4 == 0 and nxt.ld % 4 == 0 and mean is not None
                    and ops.tc_supported(M, sp.cin, sp.cout, ldg, sp.cin)):
                lazy = (nxt.raw, nxt.ld, nxt.scale, nxt.shift, nxt.relu, mean, var, s12, eps, True)
            else:
                out = G if (own_g and ldg == C) else None
                dY = ops.act_bwd_apply(G, ldg, nxt.raw, nxt.ld, nxt.scale, nxt.shift, mean, var, eps,
                                       nxt.relu, True, s1, s2, M, C, out=out, ldo=C)
        elif sp.relu:
            out = G if (own_g and ldg == C) else None
            dY = ops.act_bwd_apply(G, ldg, nxt.raw, nxt.ld, None, None, None, None, 0.0, True,
                                   False, None, None, M, C, out=out, ldo=C)
        else:
            dY, ldy = G, ldg
        red = None

        # weight gradient: dW[cout, cin] = dY^T [cout, M] * act(prev)[M, cin]
        def weight_grads(dY, ldy, cur=cur, nxt=nxt, mean=mean, sp=sp, Wp=Wp, C=C):
            kpad = _padded_k(sp.cin, cur.ld)
            if ops.tc_dw_supported(M, sp.cout, kpad, ldy, cur.ld) and (kpad == sp.cin or not cur.pending):
                dW = ops.tc_dw(dY, ldy, cur.raw, cur.ld, M, sp.cout, kpad, p_aff=cur.aff())
                if kpad != sp.cin:
                    dW = dW[:, :sp.cin].contiguous()
            else:
                dW = ops.gemm(dY, ldy, False, cur.raw, cur.ld, False, sp.cout, sp.cin, M, b_aff=cur.aff())
            db = None
            if sp.b is not None:
                if sp.bn is not None and nxt.scale is not None and mean is not None:
                    # a bias that feeds a batch-statistics BatchNorm has an analytically zero
                    # gradient (sum_m dY = -scale*s2/M * sum_m xhat = 0); the reference holds
                    # rounding noise there.  No reduction is launched.
                    db = _zeros(C, dY.device)
                else:
                    db = ops.colsum(dY, ldy, M, C)
            return dW.view(Wp.shape), db

        def run_weight_grads(dY, ldy):
            side = ops.SIDE[0]
            if side is None:
                grads[sp.w], db = weight_grads(dY, ldy)
                if sp.b is not None:
                    grads[sp.b] = db
            else:
                # Trainer mode: nothing downstream reads a weight gradient, so it runs on the side
                # stream while this stream goes on with the data gradient and the next layer.  The
                # result goes straight to .grad (see _RecurrentECCFunction.backward).
                with side.fork(dY, saved[li]):
                    dW, db = weight_grads(dY, ldy)
                    _accumulate_grad(Wp, dW)
                    if sp.b is not None:
                        if db is _ZEROS.get((C, dY.device.index)):
                            db = db.clone()  # .grad must not alias the shared zero vector
                        _accumulate_grad(params[sp.b], db)

        if lazy is None:
            run_weight_grads(dY, ldy)  # forked before the data gradient: the side stream starts earlier
        Gn = None
        if want_dx:
            if lazy is not None or ops.tc_supported(M, sp.cin, sp.cout, ldy, sp.cin):
                bnred = None
                if (ops.USE_FUSED_BNBWD[0] and li > 0 and specs[li - 1].bn is not None
                        and saved[li - 1][2] is not None and cur.ld % 4 == 0):
                    # `cur` is the layer below's deferred output: its raw y, BatchNorm fold and ReLU
                    bnred = (cur.raw, cur.ld, cur.scale, cur.shift, saved[li - 1][2], saved[li - 1][3],
                             specs[li - 1].bn.eps, cur.relu)
                res = ops.tc_gemm(G if lazy is not None else dY, ldg if lazy is not None else ldy,
                                  _w2d(Wp), sp.cin, True, M, sp.cin, sp.cout, bnbwd=lazy, bnred=bnred)
                res = list(res) if isinstance(res, tuple) else [res]
                Gn = res.pop(0)
                if lazy is not None:
                    dY, ldy = res.pop(0), C
                if bnred is not None:
                    red = res.pop(0)
            else:
                Gn = ops.gemm(dY, ldy, True, _w2d(Wp), sp.cin, False, M, sp.cin, sp.cout)
        elif lazy is not None:  # (cannot happen: lazy implies want_dx)
            raise AssertionError
        if lazy is not None:
            run_weight_grads(dY, ldy)
        if want_dx:
            G, ldg, own_g = Gn, sp.cin, True
        else:
            G = None
    return G


def pack_jobs(specs, params, M, ld_in, need_input_grad):
    """Weight images a chain over M rows will ask for (same selection rules as chain_forward /
    chain_backward), as jobs for ops.prepack."""
    jobs = []
    ld = ld_in
    for li, sp in enumerate(specs):
        W = _w2d(params[sp.w])
        kpad = _padded_k(sp.cin, ld)
        if ops.tc_supported(M, sp.cout, kpad, ld, sp.cout):
            jobs.append((W, sp.cin, False, sp.cout, kpad, sp.cin))
        if (li > 0 or need_input_grad) and ops.tc_supported(M, sp.cin, sp.cout, sp.cout, sp.cin):
            jobs.append((W, sp.cin, True, sp.cin, sp.cout, sp.cout))
        ld = sp.cout
    return jobs


class ChainFunction(torch.autograd.Function):
    """autograd wrapper: y = chain(x) with the final activation materialised."""

    @staticmethod
    def forward(ctx, x, specs, training, *params):
        x = x.contiguous()
        M, K = x.shape
        saved = [] if training else None  # eval-mode forwards keep nothing (no backward)
        out = chain_forward(Deferred(x, K, K), M, specs, params, training, saved)
        y = out.materialise(M)
        ctx.specs, ctx.saved, ctx.M = specs, saved, M
        ctx.nparams = len(params)
        ctx.params = params
        return y

    @staticmethod
    def backward(ctx, gy):
        if ctx.saved is None:
            raise RuntimeError("backward through an eval-mode forward is not supported "
                               "(the reference never does it: learning/main.py:229-311)")
        gy = gy.contiguous()
        grads = [None] * ctx.nparams
        gx = chain_backward(gy, gy.shape[1], ctx.M, ctx.specs, ctx.params, ctx.saved,
                            ctx.needs_input_grad[0], grads)
        ctx.saved = None
        return (gx, None, None) + tuple(grads)


def run_sequential(seq, x, training):
    """Runs an nn.Sequential of Linear/BN/ReLU through the fused chain with autograd support."""
    specs, params = parse_sequential(seq, training)
    return ChainFunction.apply(x, specs, training, *params)
