"""Typed Python wrappers over the C-ABI (include/spg_b200.h).

Every function takes CUDA tensors, validates shape/dtype/contiguity on the host and enqueues
on torch's current stream.  CPU tensors are rejected: there is no CPU implementation in the
product (the CPU restatement lives in oracle/ and is test infrastructure only).
"""
import os
import weakref

import numpy as np
import torch

from . import _lib

F32, F64 = 0, 1
GRU_LAYERNORM, GRU_INGATE, GRU_BIAS = 1, 2, 4


def _need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError(
                "superpoint_graph_b200 ops run on sm_100a CUDA tensors only (got a CPU tensor); "
                "there is no CPU fallback")


def _dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise TypeError("unsupported dtype %s" % t.dtype)


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


_workspaces = {}
_retired_workspaces = []  # outgrown buffers are never freed: a captured CUDA graph may hold their address


def workspace(nfloats, device, slot=0):
    """Per (device, stream, slot) scratch buffer; stream order makes reuse across calls safe.
    Slots keep buffers that are live in the SAME kernel apart (0: split-K / partial products,
    1: statistics partials).  A buffer that has to grow is replaced by one at least twice as large
    and the old one is kept alive for the life of the process (Trainer.capture bakes workspace
    addresses into CUDA graphs; geometric growth bounds the retired total by the final size)."""
    key = (device.index, _lib.current_stream(), slot)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nfloats:
        grow = 0 if buf is None else 2 * buf.numel()
        if buf is not None:
            _retired_workspaces.append(buf)
        buf = torch.empty(max(int(nfloats), grow, 1 << 16), dtype=torch.float32, device=device)
        _workspaces[key] = buf
    return buf


def zero_(t):
    _need_cuda(t)
    assert t.is_contiguous()
    _lib.call("spg_zero", t, t.numel() * t.element_size(), _lib.current_stream())
    return t


# ------------------------------------------------------------------ graph structure
class EccGraph(object):
    """Device-side CSR views of one batched graph, shared by all ECC kernels.

    Derived from the reference's `(idxn, idxe, degs)` triple (ref: learning/ecc/GraphConvInfo.py:48-69):
    `tgt_rowptr` is the exclusive scan of the in-degrees, `edge_tgt` the target of every edge,
    `(src_rowptr, src_perm)` a stable source-sorted CSR used by the atomic-free grad_input kernel.
    CUDA inputs: `EccGraph.from_device` (spg_graph_build, on the device); host inputs: this constructor
    (numpy), which the CPU tests pin and the GPU tests compare the device builder with, bit for bit.
    """

    def __init__(self, idxn, idxe, degs, n_in=None):
        idxn_np = idxn.detach().cpu().numpy().astype(np.int64, copy=False)
        degs_np = degs.detach().cpu().numpy().astype(np.int64, copy=False)
        self.n_out = int(degs_np.shape[0])
        self.n_edges = int(idxn_np.shape[0])
        if int(degs_np.sum()) != self.n_edges:
            raise ValueError("sum(degs)=%d does not match the number of edges %d"
                             % (int(degs_np.sum()), self.n_edges))
        if n_in is None:
            n_in = max(self.n_out, int(idxn_np.max()) + 1 if self.n_edges else 0)
        self.n_in = int(n_in)
        if self.n_edges and (idxn_np.min() < 0 or idxn_np.max() >= self.n_in):
            raise ValueError("idxn out of range")
        host = build_csr_host(idxn_np, degs_np, self.n_in)
        self.host = host
        self.idxe_host = None if idxe is None else idxe.detach().cpu().numpy().astype(np.int32)
        self._dev = {}

    GRAPH_FIELDS = ("tgt_rowptr", "idxn", "edge_tgt", "src_rowptr", "src_perm")

    @classmethod
    def from_device(cls, idxn, degs, n_in=None, check=True, idxe=None):
        """Builds the views ON THE DEVICE from the reference's collated pair (int64 CUDA tensors, as
        GraphConvInfo.cuda() holds them, GraphConvInfo.py:71-77) — spg_graph_build: a scan, a stable radix
        sort and three small kernels instead of host numpy; bit-identical to the host builder.
        check=True reads the device status word back (one synchronisation) and raises like the host
        builder does; callers that validated the host arrays already pass check=False."""
        _need_cuda(idxn, degs)
        g = cls.__new__(cls)
        g.n_out, g.n_edges = int(degs.numel()), int(idxn.numel())
        g.n_in = int(n_in if n_in is not None else g.n_out)
        g.host, g.idxe_host = None, None
        dev = graph_build_alloc(g.n_out, g.n_in, g.n_edges, idxn.device)
        graph_build_into(dev, idxn, degs, g.n_in)
        if idxe is not None:
            dev["idxe"] = idxe.to(device=idxn.device, dtype=torch.int32)
        if check:
            st = int(dev["status"].item())
            if st:
                raise ValueError("graph build rejected the arrays (status %d: 1 = idxn out of range, "
                                 "2 = bad degree, 4 = sum(degs) != number of edges)" % st)
        g._dev = {(idxn.device.type, idxn.device.index): dev}
        return g

    def to(self, device):
        device = torch.device(device)
        key = (device.type, device.index)
        if key not in self._dev:
            if self.host is None:
                raise RuntimeError("this graph was built on %s; it has no host copy to move" % (list(self._dev),))
            d = {k: torch.from_numpy(v).to(device) for k, v in self.host.items()}
            d["idxe"] = None if self.idxe_host is None else torch.from_numpy(self.idxe_host).to(device)
            self._dev[key] = d
        return self._dev[key]


def graph_build_alloc(n_out, n_in, n_edges, device):
    """Output tensors + status word + workspace of spg_graph_build (static addresses: a captured CUDA graph
    reads them, HostBatch.copy_into rebuilds into them)."""
    nbytes = torch.zeros(1, dtype=torch.int64)
    _lib.call("spg_graph_build_workspace", n_out, n_in, n_edges, nbytes)
    i32 = dict(dtype=torch.int32, device=device)
    return {"tgt_rowptr": torch.empty(n_out + 1, **i32), "idxn": torch.empty(n_edges, **i32),
            "edge_tgt": torch.empty(n_edges, **i32), "src_rowptr": torch.empty(n_in + 1, **i32),
            "src_perm": torch.empty(n_edges, **i32), "idxe": None, "status": torch.zeros(1, **i32),
            "_ws": torch.empty(int(nbytes[0]) + 256, dtype=torch.uint8, device=device)}


def graph_build_into(dev, idxn, degs, n_in):
    """Runs spg_graph_build on the current stream into the tensors of graph_build_alloc()."""
    _need_cuda(idxn, degs)
    assert idxn.dtype == torch.int64 and degs.dtype == torch.int64 and idxn.is_contiguous() and degs.is_contiguous()
    ws = dev["_ws"]
    off = (-ws.data_ptr()) % 256
    _lib.call("spg_graph_build", idxn, degs, degs.numel(), int(n_in), idxn.numel(), dev["idxn"], dev["tgt_rowptr"],
              dev["edge_tgt"], dev["src_rowptr"], dev["src_perm"], dev["status"], ws.data_ptr() + off,
              ws.numel() - off, _lib.current_stream())


def build_csr_host(idxn, degs, n_in):
    """Pure-numpy structure builder (also exercised by the CPU tests)."""
    n_edges = idxn.shape[0]
    tgt_rowptr = np.zeros(degs.shape[0] + 1, dtype=np.int64)
    np.cumsum(degs, out=tgt_rowptr[1:])
    edge_tgt = np.repeat(np.arange(degs.shape[0], dtype=np.int64), degs)
    src_perm = np.argsort(idxn, kind="stable")
    src_counts = np.bincount(idxn, minlength=n_in) if n_edges else np.zeros(n_in, dtype=np.int64)
    src_rowptr = np.zeros(n_in + 1, dtype=np.int64)
    np.cumsum(src_counts, out=src_rowptr[1:])
    if n_edges >= 2 ** 31 or n_in >= 2 ** 31:
        raise ValueError("graph too large for int32 indices")
    return {
        "tgt_rowptr": tgt_rowptr.astype(np.int32),
        "idxn": idxn.astype(np.int32),
        "edge_tgt": edge_tgt.astype(np.int32),
        "src_rowptr": src_rowptr.astype(np.int32),
        "src_perm": src_perm.astype(np.int32),
    }


# ------------------------------------------------------------------------------ ECC
def ecc_fwd(x, w, graph, c_out, out=None):
    _need_cuda(x, w)
    x, w = _c(x), _c(w)
    g = graph.to(x.device)
    is_mat = int(w.dim() == 3)
    c_in = x.shape[1]
    if x.shape[0] != graph.n_in:
        raise ValueError("input has %d rows, graph has %d nodes" % (x.shape[0], graph.n_in))
    n_w = g["idxe"].max().item() + 1 if g["idxe"] is not None else graph.n_edges
    if w.shape[0] < n_w:
        raise ValueError("weights has %d rows, graph needs %d" % (w.shape[0], n_w))
    if out is None:
        out = torch.empty((graph.n_out, c_out), dtype=x.dtype, device=x.device)
    _lib.call("spg_ecc_fwd", x, w, g["tgt_rowptr"], g["idxn"], g["idxe"], out, graph.n_out,
              graph.n_edges, c_in, c_out, is_mat, _dt(x), _lib.current_stream())
    return out


def ecc_bwd_w(xs, gs, graph, w_shape, n_iter=1, out=None, accumulate=False):
    """xs: [n_iter, n_in, c_in] (or [n_in, c_in]); gs: [n_iter, n_out, c_out]."""
    _need_cuda(xs, gs)
    xs, gs = _c(xs), _c(gs)
    g = graph.to(xs.device)
    is_mat = int(len(w_shape) == 3)
    c_in, c_out = xs.shape[-1], gs.shape[-1]
    if out is None:
        if g["idxe"] is not None:
            out = torch.zeros(w_shape, dtype=xs.dtype, device=xs.device)
        else:
            out = torch.empty(w_shape, dtype=xs.dtype, device=xs.device)
    x_stride = xs.shape[-2] * c_in if xs.dim() == 3 else 0
    g_stride = gs.shape[-2] * c_out if gs.dim() == 3 else 0
    _lib.call("spg_ecc_bwd_w", xs, gs, x_stride, g_stride, n_iter, g["tgt_rowptr"], g["idxn"],
              g["idxe"], g["edge_tgt"], out, graph.n_out, graph.n_edges, c_in, c_out, is_mat,
              int(accumulate), _dt(xs), _lib.current_stream())
    return out


def ecc_bwd_x(w, g_out, graph, c_in, add0=None, add1=None):
    _need_cuda(w, g_out, add0, add1)
    w, g_out = _c(w), _c(g_out)
    add0 = None if add0 is None else _c(add0)
    add1 = None if add1 is None else _c(add1)
    g = graph.to(w.device)
    is_mat = int(w.dim() == 3)
    c_out = g_out.shape[1]
    gx = torch.empty((graph.n_in, c_in), dtype=w.dtype, device=w.device)
    _lib.call("spg_ecc_bwd_x", w, g_out, g["tgt_rowptr"], g["src_rowptr"], g["src_perm"],
              g["edge_tgt"], g["idxe"], add0, add1, gx, graph.n_in, graph.n_edges, c_in, c_out,
              is_mat, _dt(w), _lib.current_stream())
    return gx


# ------------------------------------------------------------------------------ GRU
def gru_fwd(x, h, w_ih, w_hh, b_ih, b_hh, w_ig, b_ig, flags, out=None):
    _need_cuda(x, h, w_ih, w_hh)
    x, h = _c(x), _c(h)
    n, H = h.shape
    assert x.shape == h.shape and w_ih.shape == (3 * H, H) and w_hh.shape == (3 * H, H)
    if out is None:
        out = torch.empty_like(h)
    _lib.call("spg_gru_fwd", x, h, _c(w_ih), _c(w_hh), b_ih, b_hh,
              None if w_ig is None else _c(w_ig), b_ig, out, n, H, flags, _lib.current_stream())
    return out


def gru_bwd(x, h, gy, w_ih, w_hh, b_ih, b_hh, w_ig, b_ig, flags, d_gi, d_gh, d_q, xprime, dpre,
            d_x=None, d_h=None):
    _need_cuda(x, h, gy)
    x, h, gy = _c(x), _c(h), _c(gy)
    n, H = h.shape
    if d_x is None:
        d_x = torch.empty_like(h)
    if d_h is None:
        d_h = torch.empty_like(h)
    _lib.call("spg_gru_bwd", x, h, gy, _c(w_ih), _c(w_hh), b_ih, b_hh,
              None if w_ig is None else _c(w_ig), b_ig, d_x, d_h, d_gi, d_gh, d_q, xprime, dpre,
              n, H, flags, _lib.current_stream())
    return d_x, d_h


def rnn_vv_supported(weights, graph, n, H):
    """True when the fused recurrence kernels apply (vector filters, H == 32, no idxe, training-batch
    sizes); everything else runs the per-step kernels."""
    return (USE_FUSED_RNN[0] and weights.dim() == 2 and weights.dtype == torch.float32
            and graph.idxe_host is None and graph.n_in == n and graph.n_out == n
            and bool(_lib.lib().spg_rnn_vv_supported(n, H)))


def rnn_vv_fwd(hs, inps, weights, graph, cell, flags):
    """hs [R+1,n,H] with hs[0] set, inps [R,n,H]; fills hs[1:], inps (ref: learning/modules.py:160-180)."""
    _need_cuda(hs, inps, weights)
    R, n, H = inps.shape
    g = graph.to(hs.device)
    w_ih, w_hh, b_ih, b_hh, w_ig, b_ig = cell
    bar = torch.empty(4, dtype=torch.int32, device=hs.device)
    _lib.call("spg_rnn_vv_fwd", hs, inps, _c(weights), g["tgt_rowptr"], g["idxn"], _c(w_ih), _c(w_hh),
              b_ih, b_hh, None if w_ig is None else _c(w_ig), b_ig, n, H, R, flags, bar,
              _lib.current_stream())


def rnn_vv_bwd(hs, inps, weights, graph, cell, flags, gtop, gcat, ginp, d_gi, d_gh, d_q, xp, dpre):
    """Backward of rnn_vv_fwd; returns the gradient w.r.t. hs[0]."""
    _need_cuda(hs, inps, weights, gtop)
    R, n, H = inps.shape
    g = graph.to(hs.device)
    w_ih, w_hh, b_ih, b_hh, w_ig, b_ig = cell
    bar = torch.empty(4, dtype=torch.int32, device=hs.device)
    dh = torch.empty((n, H), dtype=torch.float32, device=hs.device)
    gh0 = torch.empty((n, H), dtype=torch.float32, device=hs.device)
    _lib.call("spg_rnn_vv_bwd", hs, inps, _c(weights), gtop, gcat, g["tgt_rowptr"], g["src_rowptr"],
              g["src_perm"], g["edge_tgt"], _c(w_ih), _c(w_hh), b_ih, b_hh,
              None if w_ig is None else _c(w_ig), b_ig, ginp, dh, gh0, d_gi, d_gh, d_q, xp, dpre,
              n, H, R, flags, bar, _lib.current_stream())
    return gh0


# ---------------------------------------------------------------------------- dense
GEMM_TRACE = None  # set to [] to record (description, start, end) events of every SIMT gemm call
GEMM_FLOPS = [0]  # algorithmic FLOPs (2*M*N*K) issued through gemm(); read by bench.py


def _auto_split(M, N, K):
    tiles = ((M + 127) // 128) * ((N + 63) // 64)
    if tiles >= 148 or K < 256:
        return 1
    split = min((2 * 148 + tiles - 1) // tiles, max(1, K // 64))
    return max(1, split)


def _merge_stats(sws, tiles, N, M, dev, fold):
    """(mean, var) or, with fold=(gamma, beta, eps, rm, rv, nbt, momentum), (mean, var, scale, shift)."""
    mean = torch.empty(N, dtype=torch.float32, device=dev)
    var = torch.empty(N, dtype=torch.float32, device=dev)
    if fold is None:
        _lib.call("spg_colstats_merge", sws, tiles, N, mean, var, _lib.current_stream())
        return mean, var
    gamma, beta, eps, rm, rv, nbt, mom = fold
    scale = torch.empty(N, dtype=torch.float32, device=dev)
    shift = torch.empty(N, dtype=torch.float32, device=dev)
    _lib.call("spg_colstats_merge_fold", sws, tiles, N, mean, var, gamma, beta, float(eps), scale, shift,
              rm, rv, nbt, float(mom), int(M), _lib.current_stream())
    return mean, var, scale, shift


def gemm(A, lda, a_kmajor, B, ldb, b_kmajor, M, N, K, bias=None, out=None, ldc=None,
         a_aff=None, b_aff=None, split_k=None, stats=False, fold=None):
    """C[M,N] = opA(A) opB(B) + bias.  a_aff/b_aff = (scale|None, shift|None, relu)."""
    _need_cuda(A, B)
    dev = A.device
    if out is None:
        out = torch.empty((M, N), dtype=torch.float32, device=dev)
        ldc = N
    elif ldc is None:
        ldc = out.stride(0)
    a_s, a_t, a_r = a_aff if a_aff is not None else (None, None, False)
    b_s, b_t, b_r = b_aff if b_aff is not None else (None, None, False)
    GEMM_FLOPS[0] += 2 * M * N * K
    if GEMM_TRACE is not None:
        ev0 = torch.cuda.Event(enable_timing=True)
        ev0.record()
    if split_k is None:
        split_k = 1 if stats else _auto_split(M, N, K)
    ws = workspace(split_k * M * N, dev) if split_k > 1 else None
    tiles = (M + 127) // 128
    sws = workspace((tiles + tiles // 256 + 2) * N * 3, dev, slot=1) if stats else None
    _lib.call("spg_gemm", A, lda, int(a_kmajor), B, ldb, int(b_kmajor), bias, out, ldc, M, N, K,
              a_s, a_t, int(bool(a_r)), b_s, b_t, int(bool(b_r)), split_k, ws, sws,
              _lib.current_stream())
    if GEMM_TRACE is not None:
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        GEMM_TRACE.append(("M=%d N=%d K=%d a%d b%d split=%d" % (M, N, K, int(a_kmajor), int(b_kmajor), split_k),
                           ev0, ev1))
    if stats:
        return (out,) + _merge_stats(sws, tiles, N, M, dev, fold)
    return out


USE_TC = [os.environ.get("SPG_TC", "1") != "0"]  # tcgen05 path for the large point-wise layers
USE_FUSED_RNN = [os.environ.get("SPG_FUSED_RNN", "1") != "0"]  # one-kernel R x {ECC, cell} loop
USE_FUSED_BNBWD = [os.environ.get("SPG_FUSED_BNBWD", "1") != "0"]  # BatchNorm backward inside the dX GEMM (prologue + epilogue sums)
USE_FUSED_EVAL = [os.environ.get("SPG_FUSED_EVAL", "1") != "0"]  # eval-mode PointNet trunk as one kernel per chain
def set_pdl(mode):
    """Programmatic dependent launch policy of the library (spg_set_pdl): 1 = every kernel is scheduled while
    its predecessor on the stream still runs and waits on the device for it (measured -1.5 ... -4.5 % on the
    single-stream inference workloads), 0 = plain stream order (the two-stream training schedule is 2 % faster
    that way: early-resident GEMM CTAs take SMs from the weight-gradient stream).  An explicit SPG_PDL in the
    environment wins."""
    if "SPG_PDL" not in os.environ:
        _lib.call("spg_set_pdl", int(mode))


USE_SIDE_STREAM = [os.environ.get("SPG_SIDE_STREAM", "1") != "0"]  # Trainer: block-local weight gradients on a 2nd stream


def tc_supported(M, N, K, lda=0, ldc=0):
    return (USE_TC[0] and M >= 512 and lda % 4 == 0 and ldc % 4 == 0
            and bool(_lib.lib().spg_tc_gemm_supported(int(M), int(N), int(K))))


PACK_CACHE = {}   # (W ptr, ldw, transpose, N, K, k_valid) -> image, valid until the weights change
_PACK_TABLES = {}  # tuple of job keys -> (device table, images, total)
PACK_LEARN = [None]  # dict owned by a Trainer: images packed on demand in its step, batched from the next step on


def prepack(jobs):
    """Packs the weight images of many layers with ONE launch and publishes them in PACK_CACHE.
    jobs: [(W, ldw, transpose, N, K, k_valid)].  The caller clears PACK_CACHE when the weights
    change (Trainer does after every backward)."""
    if not jobs:
        return
    keys = tuple((W.data_ptr(), int(ldw), int(bool(tr)), int(N), int(K), int(kv)) for W, ldw, tr, N, K, kv in jobs)
    ent = _PACK_TABLES.get(keys)
    dev = jobs[0][0].device
    if ent is None:
        rows, imgs, total = [], [], 0
        for (ptr, ldw, tr, N, K, kv) in keys:
            img = torch.empty(2 * N * K, dtype=torch.float32, device=dev)
            imgs.append(img)
            rows.append([ptr, ldw, tr, N, K, kv, img.data_ptr(), total])
            total += N * K
        table = torch.tensor(rows, dtype=torch.int64).to(dev)
        ent = _PACK_TABLES[keys] = (table, imgs, total)
    table, imgs, total = ent
    _lib.call("spg_tc_pack_weights_multi", table, len(keys), total, _lib.current_stream())
    for k, img in zip(keys, imgs):
        PACK_CACHE[k] = img


def _weight_image(W, ldw, transpose, N, K, kv, dev):
    key = (W.data_ptr(), int(ldw), int(bool(transpose)), int(N), int(K), int(kv))
    img = PACK_CACHE.get(key)
    if img is None:
        img = torch.empty(2 * N * K, dtype=torch.float32, device=dev)
        _lib.call("spg_tc_pack_weights", W, ldw, int(bool(transpose)), N, K, kv, img, _lib.current_stream())
        if PACK_LEARN[0] is not None:
            PACK_LEARN[0][key] = (W, int(ldw), bool(transpose), int(N), int(K), kv)
    return img


def tc_gemm(A, lda, W, ldw, transpose, M, N, K, bias=None, a_aff=None, stats=False, k_valid=None,
            fold=None, bnbwd=None, bnred=None):
    """C[M,N] = f(A)[M,K] B[N,K]^T + bias on the tcgen05 3xTF32 kernel (spg_tc_gemm_ex).
    transpose=False: B = W ([N,K], ld ldw); True: B = W^T with W [K,N].

    stats / fold: batch statistics of C (and the BatchNorm fold) finished inside the kernel; returns
        (C, mean, var[, scale, shift]).
    bnbwd = (Y, ldy, scale, shift, relu, mean, var, s12, eps, want_dy): A is dL/d(activation) of a
        BatchNorm+ReLU layer whose raw output is Y; the prologue turns it into dL/dY on the fly.
        With want_dy the kernel also stores dL/dY [M,K] (for the weight-gradient kernel).
    bnred = (Y2, ldy2, scale2, shift2, mean2, var2, eps2, relu2): C is dL/d(activation) of the layer
        below; its BatchNorm-backward sums s1|s2 [2N] come out of the epilogue.
    Returns C, or a tuple (C, [mean, var, [scale, shift]], [dY], [s12]) in that order."""
    _need_cuda(A, W)
    dev = A.device
    kv = int(K if k_valid is None else k_valid)
    img = _weight_image(W, ldw, transpose, N, K, kv, dev)
    out = torch.empty((M, N), dtype=torch.float32, device=dev)
    a_s, a_t, a_r = a_aff if a_aff is not None else (None, None, False)
    a2 = a_mean = a_var = a_s12 = dy = None
    lda2 = lddy = 0
    a_eps = 0.0
    if bnbwd is not None:
        a2, lda2, a_s, a_t, a_r, a_mean, a_var, a_s12, a_eps, want_dy = bnbwd
        if want_dy:
            dy = torch.empty((M, K), dtype=torch.float32, device=dev)
            lddy = K
    epi, ws = 0, None
    mean = var = scale = shift = gamma = beta = rm = rv = nbt = None
    eps = mom = 0.0
    e = (None, 0, None, None, None, None, 0.0, False)
    s12 = None
    if stats:
        epi = 1
        mean = torch.empty(N, dtype=torch.float32, device=dev)
        var = torch.empty(N, dtype=torch.float32, device=dev)
        if fold is not None:
            gamma, beta, eps, rm, rv, nbt, mom = fold
            scale = torch.empty(N, dtype=torch.float32, device=dev)
            shift = torch.empty(N, dtype=torch.float32, device=dev)
    elif bnred is not None:
        epi = 2
        e = bnred
        s12 = torch.empty(2 * N, dtype=torch.float32, device=dev)
    if epi:
        ws = workspace(MAX_TC_PARTIALS[0] * N * 3, dev, slot=1)
    GEMM_FLOPS[0] += 2 * M * N * K
    TC_FLOPS[0] += 2 * M * N * K
    _lib.call("spg_tc_gemm_ex", A, lda, img, bias, out, N, M, N, K, a_s, a_t, int(bool(a_r)),
              a2, lda2, a_mean, a_var, a_s12, float(a_eps), dy, lddy, epi, ws,
              mean, var, gamma, beta, float(eps), scale, shift, rm, rv, nbt, float(mom),
              e[0], e[1], e[2], e[3], e[4], e[5], float(e[6]), int(bool(e[7])), s12,
              _lib.current_stream())
    res = [out]
    if stats:
        res += [mean, var] + ([scale, shift] if fold is not None else [])
    if dy is not None:
        res.append(dy)
    if s12 is not None:
        res.append(s12)
    return res[0] if len(res) == 1 else tuple(res)


MAX_TC_PARTIALS = [148]  # spg_tc_gemm_max_partials(): CTAs along the rows = partials per column

TC_FLOPS = [0]  # algorithmic FLOPs through tc_gemm (forward + data gradients)
DW_FLOPS = [0]  # algorithmic FLOPs through tc_dw (weight gradients)


def tc_dw_supported(M, co, ci, lddy, ldp):
    return (USE_TC[0] and M >= 2048 and lddy % 4 == 0 and ldp % 4 == 0
            and bool(_lib.lib().spg_tc_dw_supported(int(M), int(co), int(ci))))


def tc_dw(dY, lddy, P, ldp, M, co, ci, p_aff=None):
    """dW[co,ci] = dY^T [co,M] f(P)[M,ci] on the tcgen05 3xTF32 kernel (ci may be the padded
    leading dimension of P; the caller slices the valid columns)."""
    _need_cuda(dY, P)
    dev = dY.device
    ctas = int(_lib.lib().spg_tc_dw_ctas(int(M)))
    ws = workspace(ctas * co * ci, dev)
    out = torch.empty((co, ci), dtype=torch.float32, device=dev)
    p_s, p_t, p_r = p_aff if p_aff is not None else (None, None, False)
    GEMM_FLOPS[0] += 2 * M * co * ci
    DW_FLOPS[0] += 2 * M * co * ci
    _lib.call("spg_tc_dw", dY, lddy, P, ldp, p_s, p_t, int(bool(p_r)), out, ws, M, co, ci,
              _lib.current_stream())
    return out


def _chunks(M):
    return max(1, (M + 255) // 256)


def colstats(Y, ldy, M, C):
    _need_cuda(Y)
    mean = torch.empty(C, dtype=torch.float32, device=Y.device)
    var = torch.empty(C, dtype=torch.float32, device=Y.device)
    ws = workspace(3 * C * (_chunks(M) + _chunks(M) // 256 + 2), Y.device)
    _lib.call("spg_colstats", Y, ldy, M, C, mean, var, ws, _lib.current_stream())
    return mean, var


def bn_fold(mean, var, gamma, beta, eps, running_mean=None, running_var=None, momentum=0.1, M=0,
            num_batches_tracked=None):
    _need_cuda(mean, var)
    C = mean.numel()
    scale = torch.empty(C, dtype=torch.float32, device=mean.device)
    shift = torch.empty(C, dtype=torch.float32, device=mean.device)
    _lib.call("spg_bn_fold", mean, var, gamma, beta, float(eps), scale, shift, running_mean,
              running_var, num_batches_tracked, float(momentum), int(M), C, _lib.current_stream())
    return scale, shift


def affine_act(Y, ldy, M, C, scale=None, shift=None, relu=False, out=None, ldo=None):
    _need_cuda(Y)
    if out is None:
        out = torch.empty((M, C), dtype=torch.float32, device=Y.device)
        ldo = C
    _lib.call("spg_affine_act", Y, ldy, scale, shift, int(bool(relu)), out, ldo, M, C,
              _lib.current_stream())
    return out


def colsum(X, ldx, M, C):
    _need_cuda(X)
    out = torch.empty(C, dtype=torch.float32, device=X.device)
    ws = workspace(C * _chunks(M), X.device)
    _lib.call("spg_colsum", X, ldx, M, C, out, ws, _lib.current_stream())
    return out


def act_bwd_reduce(G, ldg, Y, ldy, scale, shift, mean, var, eps, relu, M, C):
    _need_cuda(G, Y)
    """-> s12 [2C]: s1 = s12[:C] (sum of the masked gradient), s2 = s12[C:] (same, weighted by xhat)."""
    s12 = torch.empty(2 * C, dtype=torch.float32, device=G.device)
    s1, s2 = s12[:C], s12[C:]  # contiguous pair: one merge launch writes both
    ws = workspace(2 * C * _chunks(M), G.device)
    _lib.call("spg_act_bwd_reduce", G, ldg, Y, ldy, scale, shift, mean, var, float(eps),
              int(bool(relu)), s1, s2, ws, M, C, _lib.current_stream())
    return s12


def act_bwd_apply(G, ldg, Y, ldy, scale, shift, mean, var, eps, relu, has_bn, s1, s2, M, C,
                  out=None, ldo=None):
    _need_cuda(G)
    if out is None:
        out = torch.empty((M, C), dtype=torch.float32, device=G.device)
        ldo = C
    _lib.call("spg_act_bwd_apply", G, ldg, Y, ldy, scale, shift, mean, var, float(eps),
              int(bool(relu)), int(bool(has_bn)), s1, s2, out, ldo, M, C, _lib.current_stream())
    return out


# ------------------------------------------------------------------------- PointNet
def cloud_rows(clouds, T, ld, add_eye=False):
    _need_cuda(clouds, T)
    clouds = _c(clouds)
    B, F, L = clouds.shape
    rows = torch.empty((B * L, ld), dtype=torch.float32, device=clouds.device)
    _lib.call("spg_cloud_rows", clouds, None if T is None else _c(T), int(bool(add_eye)), rows, ld,
              B, F, L, _lib.current_stream())
    return rows


def rows_to_clouds(rows, ld, B, F, L):
    _need_cuda(rows)
    out = torch.empty((B, F, L), dtype=torch.float32, device=rows.device)
    _lib.call("spg_rows_to_clouds", rows, ld, out, B, F, L, _lib.current_stream())
    return out


def segmax_fwd(Y, ldy, B, L, C, scale, shift, relu, pooled, ldp):
    _need_cuda(Y, pooled)
    argmax = torch.empty((B, C), dtype=torch.int32, device=Y.device)
    _lib.call("spg_segmax_fwd", Y, ldy, scale, shift, int(bool(relu)), pooled, ldp, argmax, B, L, C,
              _lib.current_stream())
    return argmax


def segmax_bwd(g_pooled, ldg, argmax, B, L, C):
    _need_cuda(g_pooled, argmax)
    G = torch.empty((B * L, C), dtype=torch.float32, device=g_pooled.device)
    _lib.call("spg_segmax_bwd", g_pooled, ldg, argmax, G, C, B, L, C, _lib.current_stream())
    return G


def segmax_bn_bwd(g_pooled, ldg, argmax, Y, ldy, scale, shift, mean, var, eps, relu, B, L, C):
    """Fused max-pool backward + BatchNorm/ReLU backward; returns (s1, s2, dY[B*L, C])."""
    _need_cuda(g_pooled, argmax, Y)
    dev = Y.device
    s12 = torch.empty(2 * C, dtype=torch.float32, device=dev)
    dY = torch.empty((B * L, C), dtype=torch.float32, device=dev)
    ws = workspace(2 * C * ((B + 255) // 256), dev)
    _lib.call("spg_segmax_bn_bwd", g_pooled, ldg, argmax, Y, ldy, scale, shift, mean, var, float(eps),
              int(bool(relu)), s12, dY, C, ws, B, L, C, _lib.current_stream())
    return s12[:C], s12[C:], dY


def stn_apply_bwd(clouds, dXrows, ld):
    _need_cuda(clouds, dXrows)
    clouds = _c(clouds)
    B, F, L = clouds.shape
    dT = torch.empty((B, 4), dtype=torch.float32, device=clouds.device)
    _lib.call("spg_stn_apply_bwd", clouds, dXrows, ld, dT, B, F, L, _lib.current_stream())
    return dT


def rows_scatter(src, idx, n_rows_out):
    _need_cuda(src, idx)
    src = _c(src)
    n, C = src.shape
    dst = torch.empty((n_rows_out, C), dtype=torch.float32, device=src.device)
    zero_(dst)
    _lib.call("spg_rows_scatter", src, idx, dst, n, C, _lib.current_stream())
    return dst


def rows_gather(src, idx):
    _need_cuda(src, idx)
    src = _c(src)
    n = idx.numel()
    C = src.shape[1]
    dst = torch.empty((n, C), dtype=torch.float32, device=src.device)
    _lib.call("spg_rows_gather", src, idx, dst, n, C, _lib.current_stream())
    return dst


# ----------------------------------------------------------------------------- step
def ce_loss(logits, target, class_weight=None, ignore_index=-100, need_grad=True):
    _need_cuda(logits, target, class_weight)
    logits = _c(logits)
    n, C = logits.shape
    loss = torch.empty(1, dtype=torch.float32, device=logits.device)
    d_logits = torch.empty_like(logits) if need_grad else None
    ws = torch.empty(2, dtype=torch.float64, device=logits.device)
    _lib.call("spg_ce_loss", logits, _c(target), class_weight, int(ignore_index), loss, d_logits,
              ws, n, C, _lib.current_stream())
    return loss, d_logits


def clamp_adam_(param, grad, exp_avg, exp_avg_sq, step, lr, beta1=0.9, beta2=0.999, eps=1e-8,
                weight_decay=0.0, grad_clip=0.0, grad_scale=1.0):
    _need_cuda(param, grad, exp_avg, exp_avg_sq)
    _lib.call("spg_clamp_adam", param, grad, exp_avg, exp_avg_sq, param.numel(), float(lr),
              float(beta1), float(beta2), float(eps), float(weight_decay), float(grad_clip),
              float(grad_scale), int(step), _lib.current_stream())


def clamp_adam_dev_(param, grad, exp_avg, exp_avg_sq, step_counter, lr, beta1=0.9, beta2=0.999,
                    eps=1e-8, weight_decay=0.0, grad_clip=0.0, grad_scale=1.0):
    """clamp + Adam with the step count in device memory (int64 scalar tensor, incremented here)."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, step_counter)
    _lib.call("spg_clamp_adam_dev", param, grad, exp_avg, exp_avg_sq, param.numel(), float(lr),
              float(beta1), float(beta2), float(eps), float(weight_decay), float(grad_clip),
              float(grad_scale), step_counter, _lib.current_stream())


class FusedAllreduce(object):
    """Symmetric-memory plumbing of spg_allreduce_clamp_adam: a two-half staging buffer and the flag words are
    allocated with torch.distributed._symmetric_memory (CUDA VMM handles exchanged through the process
    group's store) so that every rank holds device pointers to every peer's copy over NVLink.  `grad` — the
    flat gradient the step writes — is ordinary local memory; the kernel stages it itself."""

    def __init__(self, n, device, group):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm_mem
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.grad = torch.zeros(n, dtype=torch.float32, device=device)
        self.stage = symm_mem.empty(int(_lib.lib().spg_allreduce_stage_floats(int(n))), dtype=torch.float32,
                                    device=device)
        self.stage.zero_()
        words = int(_lib.lib().spg_allreduce_flag_words(self.world))
        self.flags = symm_mem.empty(words, dtype=torch.int32, device=device)
        self.flags.zero_()
        self._h_stage = symm_mem.rendezvous(self.stage, group)
        self._h_flags = symm_mem.rendezvous(self.flags, group)
        self.stage_ptrs = int(self._h_stage.buffer_ptrs_dev)
        self.flag_ptrs = int(self._h_flags.buffer_ptrs_dev)
        self.state = torch.zeros(2, dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        dist.barrier(group=group)  # every rank's zero-fill has landed before anybody's first kernel

    def step_(self, param, exp_avg, exp_avg_sq, step_counter, lr, beta1=0.9, beta2=0.999, eps=1e-8,
              weight_decay=0.0, grad_clip=0.0):
        _need_cuda(param, exp_avg, exp_avg_sq, step_counter)
        _lib.call("spg_allreduce_clamp_adam", self.grad, self.stage_ptrs, self.flag_ptrs, self.rank, self.world,
                  param, exp_avg, exp_avg_sq, param.numel(), float(lr), float(beta1), float(beta2), float(eps),
                  float(weight_decay), float(grad_clip), 1.0 / self.world, step_counter, self.state,
                  _lib.current_stream())


USE_FUSED_ALLREDUCE = [os.environ.get("SPG_FUSED_ALLREDUCE", "1") != "0"]


# ------------------------------------------------------------------------ profiling
def prof_enable(on):
    _lib.lib().spg_prof_enable(int(on))


def prof_reset():
    _lib.lib().spg_prof_reset()


def prof_collect():
    """Returns {kernel_name: (launches, total_ms)} for kernels launched since the last reset."""
    import ctypes

    L = _lib.lib()
    L.spg_prof_collect()
    out = {}
    for k in range(L.spg_prof_num_kernels()):
        n = ctypes.c_int64(0)
        ms = ctypes.c_double(0.0)
        L.spg_prof_kernel_stats(k, ctypes.byref(n), ctypes.byref(ms))
        if n.value:
            out[L.spg_prof_kernel_name(k).decode()] = (int(n.value), float(ms.value))
    return out


def total_launches():
    return int(_lib.lib().spg_prof_total_launches())


# ------------------------------------------------------------------ side stream (Trainer only)
class SideStream(object):
    """A second stream for work nobody waits for until the gradients are gathered: the filter-net
    and cell weight gradients of the recurrent ECC block are chains of small, latency-bound kernels
    that are independent of the (large) PointNet backward which follows them on the main stream.
    `fork()` orders the side stream after everything enqueued so far, `join()` orders the current
    stream after the side stream.  Tensors handed to fork() are kept alive until join(): the
    caching allocator would otherwise recycle main-stream blocks the side kernels still read.
    Only the Trainer installs one (SIDE[0]) — a caller who does not know about join() never forks."""

    def __init__(self, device):
        self.stream = torch.cuda.Stream(device=device)
        self.keep = []
        self.active = False

    def fork(self, *keep):
        self.stream.wait_stream(torch.cuda.current_stream())
        self.keep.append(keep)
        self.active = True
        return torch.cuda.stream(self.stream)

    def join(self):
        if self.active:
            torch.cuda.current_stream().wait_stream(self.stream)
            self.active = False
        self.keep = []


SIDE = [None]


# ------------------------------------------------------------- either side of the path
def cloud_build(points, sp_start, sp_count, sample_idx, columns, n_points, normalize, xform, jitter,
                jitter_sigma, jitter_clip, seed, clouds, diameters):
    """Resample / normalise / select / augment superpoints straight into the [Nv, F, L] PointNet
    input (ref: learning/spg.py:198-260); see include/spg_b200.h spg_cloud_build."""
    _need_cuda(points, sp_start, sp_count, sample_idx, columns, xform, jitter, clouds, diameters)
    assert points.dtype == torch.float32 and points.is_contiguous()
    assert sp_start.dtype == torch.int64 and sp_count.dtype == torch.int32 and columns.dtype == torch.int32
    assert sample_idx is None or (sample_idx.dtype == torch.int32 and sample_idx.is_contiguous())
    assert xform is None or (xform.dtype == torch.float64 and xform.is_contiguous())
    assert jitter is None or (jitter.dtype == torch.float32 and jitter.is_contiguous())
    nv, F, L = clouds.shape
    assert L == n_points and columns.numel() == F
    _lib.call("spg_cloud_build", points, points.shape[1], sp_start, sp_count, sample_idx, columns, F,
              L, int(bool(normalize)), xform, jitter, float(jitter_sigma), float(jitter_clip),
              int(seed), clouds, diameters, nv, _lib.current_stream())
    return clouds, diameters


def confusion_count(logits, label_mode, label_vec, confusion, counters, want_predictions=False):
    """confusion[:, argmax(logits_i)] += label_vec[i] for the labelled nodes (ref: learning/main.py:
    257-262, metrics.py:16-18); returns the predictions of all nodes if asked."""
    _need_cuda(logits, label_mode, label_vec, confusion, counters)
    logits = _c(logits)
    label_mode, label_vec = _c(label_mode), _c(label_vec)
    n, C = logits.shape
    assert logits.dtype == torch.float32 and label_mode.dtype == torch.int64
    assert label_vec.dtype == torch.int64 and label_vec.shape == (n, C)
    assert confusion.dtype == torch.int64 and confusion.shape == (C, C) and confusion.is_contiguous()
    pred = torch.empty(n, dtype=torch.int64, device=logits.device) if want_predictions else None
    _lib.call("spg_confusion_count", logits, C, label_mode, label_vec, C, confusion, counters, pred,
              n, C, _lib.current_stream())
    return pred


def labels_to_points(labels_red, comp_ptr, point_ids, n_ver):
    _need_cuda(labels_red, comp_ptr, point_ids)
    assert labels_red.dtype == torch.int64 and comp_ptr.dtype == torch.int64 and point_ids.dtype == torch.int64
    out = torch.empty(n_ver, dtype=torch.uint8, device=labels_red.device)
    _lib.call("spg_labels_to_points", _c(labels_red), _c(comp_ptr), _c(point_ids), comp_ptr.numel() - 1, out,
              n_ver, _lib.current_stream())
    return out


def nn1_interpolate(xyz_ref, xyz_query, labels_ref=None, want_index=False):
    """Exact 1-NN (float64 distances) of every query point among the reference points."""
    _need_cuda(xyz_ref, xyz_query, labels_ref)
    assert xyz_ref.dtype == torch.float32 and xyz_query.dtype == torch.float32
    assert xyz_ref.shape[1] == 3 and xyz_query.shape[1] == 3
    xyz_ref, xyz_query = _c(xyz_ref), _c(xyz_query)
    m = xyz_query.shape[0]
    lab = torch.empty(m, dtype=torch.int64, device=xyz_ref.device) if labels_ref is not None else None
    idx = torch.empty(m, dtype=torch.int32, device=xyz_ref.device) if (want_index or labels_ref is None) else None
    _lib.call("spg_nn1_interpolate", xyz_ref, xyz_ref.shape[0], xyz_query, m,
              None if labels_ref is None else _c(labels_ref), lab, idx, _lib.current_stream())
    return lab, idx


# ------------------------------------------------------------------ ragged (CSR) superpoints
def segmax_csr_fwd(Y, ldy, offsets, C, scale, shift, relu, pooled, ldp):
    _need_cuda(Y, offsets, pooled)
    assert offsets.dtype == torch.int64 and offsets.is_contiguous()
    B = offsets.numel() - 1
    argmax = torch.empty((B, C), dtype=torch.int64, device=Y.device)
    _lib.call("spg_segmax_csr_fwd", Y, ldy, scale, shift, int(bool(relu)), offsets, pooled, ldp, argmax, B, C,
              _lib.current_stream())
    return argmax


def segmax_csr_bwd(g_pooled, ldg, argmax, P, C):
    _need_cuda(g_pooled, argmax)
    G = torch.empty((P, C), dtype=torch.float32, device=g_pooled.device)
    _lib.call("spg_segmax_csr_bwd", g_pooled, ldg, argmax, G, C, argmax.shape[0], C, P, _lib.current_stream())
    return G


def rows_xy_transform(rows, T, row_seg, add_eye=True):
    _need_cuda(rows, T, row_seg)
    assert rows.is_contiguous() and row_seg.dtype == torch.int32
    out = torch.empty_like(rows)
    _lib.call("spg_rows_xy_transform", rows, _c(T), int(bool(add_eye)), row_seg, out, rows.shape[0], rows.shape[1],
              _lib.current_stream())
    return out


def rows_xy_transform_bwd(rows, d_out, offsets):
    _need_cuda(rows, d_out, offsets)
    B = offsets.numel() - 1
    dT = torch.empty((B, 4), dtype=torch.float32, device=rows.device)
    d_out = _c(d_out)
    _lib.call("spg_rows_xy_transform_bwd", rows, rows.shape[1], d_out, d_out.shape[1], offsets, dT, B,
              _lib.current_stream())
    return dT


# ------------------------------------------------------------------ fused eval-mode PointNet trunk
def pointnet_fused_supported(F, L, widths):
    w = torch.tensor(list(widths), dtype=torch.int32)
    return USE_FUSED_EVAL[0] and bool(_lib.lib().spg_pointnet_fused_supported(int(F), int(L), len(widths), w.data_ptr()))


_FUSED_IMAGES = {}  # parameter versions -> (weight image, folded bias, widths tensor, weakrefs to the sources)
EVAL_BF16 = [False]  # eval-mode PointNet trunk in bf16 arithmetic (Trainer(dtype="bf16") sets it around eval_step)


def _root(t):
    return t if t._base is None else t._base


def pointnet_fused_image(layers, F, bf16=False):
    """layers: [(W [N,K] (2-D view), bias|None, bn_module|None)] of a Conv1d(k=1)+BatchNorm+ReLU chain in eval
    mode.  Returns (image, bias, widths): BatchNorm folded into weights and bias (scale = gamma/sqrt(rv+eps),
    bias' = bias*scale + beta - rm*scale), packed for spg_pointnet_fused_eval (fp32: tf32 hi|lo blocks of 32
    floats) or spg_pointnet_fused_eval_bf16 (bf16 blocks of 64 elements).  Cached on the tensors' addresses and
    version counters (eval weights do not change between batches).  Whoever writes these tensors behind
    torch's back (the Trainer's optimizer kernel, the running-statistics update of a training forward) bumps
    their version counters.  An entry also holds weak references to its source tensors: a tensor that died, or
    a different tensor at a recycled address with an equal version count, is a miss."""
    key, srcs = [], []
    for W, b, bn in layers:
        ts = [W, b] + ([bn.running_mean, bn.running_var, bn.weight, bn.bias] if bn is not None else [])
        key += [(x.data_ptr(), x._version) for x in ts if x is not None]
        srcs += [_root(x) for x in ts if x is not None]
    key = (int(F), bool(bf16)) + tuple(key)
    ent = _FUSED_IMAGES.get(key)
    if ent is not None and all(r() is x for r, x in zip(ent[3], srcs)):
        return ent[:3]
    dev = layers[0][0].device
    L = _lib.lib()
    widths = torch.tensor([int(W.shape[0]) for W, _, _ in layers], dtype=torch.int32)
    if bf16:
        rows = int(L.spg_pointnet_fused_bf16_image_rows(int(F), len(layers), widths.data_ptr()))
        image = torch.empty(rows * 64, dtype=torch.bfloat16, device=dev)
        kc = 64
    else:
        rows = int(L.spg_pointnet_fused_image_rows(int(F), len(layers), widths.data_ptr()))
        image = torch.empty(rows * 32, dtype=torch.float32, device=dev)
        kc = 32
    bias = torch.empty(int(widths.sum()), dtype=torch.float32, device=dev)
    row, boff, K = 0, 0, kc
    for W, b, bn in layers:
        N, kv = int(W.shape[0]), int(W.shape[1])
        scale = shift = None
        if bn is not None:
            scale, shift = bn_fold(bn.running_mean, bn.running_var, bn.weight, bn.bias, bn.eps)
        if bf16:
            _lib.call("spg_tc_pack_weights_bf16", W, W.stride(0), scale, N, K, kv, image[row * 64:],
                      _lib.current_stream())
            row += (K // 64) * N
        else:
            _lib.call("spg_tc_pack_weights_scaled", W, W.stride(0), scale, N, K, kv, image[row * 32:],
                      _lib.current_stream())
            row += (K // 32) * 2 * N
        bsl = bias[boff:boff + N]
        if b is not None:
            affine_act(b.detach().reshape(1, N), N, 1, N, scale, shift, False, out=bsl, ldo=N)
        elif shift is not None:
            bsl.copy_(shift)
        else:
            zero_(bsl)
        boff += N
        K = max(N, kc) if bf16 else N
    if len(_FUSED_IMAGES) > 64:
        _FUSED_IMAGES.clear()
    _FUSED_IMAGES[key] = (image, bias, widths, [weakref.ref(x) for x in srcs])
    return image, bias, widths


def pointnet_fused_eval(clouds, T, image, bias, widths, pooled, ldp):
    """pooled[b, :widths[-1]] = max over points of the folded conv chain on clouds[b] (xy transformed by T+I);
    the image's dtype selects the arithmetic (float32 image: 3xTF32, bfloat16 image: bf16)."""
    _need_cuda(clouds, image, bias, pooled, T)
    B, F, L = clouds.shape
    name = "spg_pointnet_fused_eval_bf16" if image.dtype == torch.bfloat16 else "spg_pointnet_fused_eval"
    _lib.call(name, clouds, B, F, L, None if T is None else _c(T), 1, image, bias,
              int(widths.numel()), widths.data_ptr(), pooled, ldp, _lib.current_stream())
    k = int(F)
    for n in widths.tolist():  # algorithmic FLOPs of the chain (valid K of the first layer, no padding)
        FUSED_FLOPS[0] += 2 * B * L * k * int(n)
        k = int(n)
    return pooled


FUSED_FLOPS = [0]  # algorithmic FLOPs through the fused eval trunk; read by bench.py
