"""The tcgen05 3xTF32 kernels of the training step (tc_gemm2.cu, tc_dw.cu, tc_pack.cu), each called through
ops, against a float64 computation on the same float32 inputs; the dense chain that strings them together
against a float64 copy of its module; and the eval path after training (folded weight images must follow
the parameters).

Errors are max|got - ref| / max|ref| per tensor.  ReLU / BatchNorm masks of the references come from the
float32 expression the kernels evaluate (fmaf(y, scale, shift) > 0, exact in float64 for float32 operands),
so a mask flip near zero cannot force a wide bound.  Bounds:
  * products (C of tc_gemm, dX, dW of tc_dw):                        PROD_TOL  = 2e-5
  * mean, scale, shift, running mean:                                 STAT_TOL  = 1e-5
  * var, running var:                                                 VAR_TOL   = 2e-5
  * BatchNorm-backward sums s1|s2 out of the GEMM epilogue:           S12_TOL   = 2e-5
  * element-wise BatchNorm backward (dY side store, segmax_bn_bwd):  STAT_TOL  = 1e-5
  * dW of tc_dw over ~1.3 M rows:                                     DW_BIG_TOL = 1e-4
  * dense chain in training mode against float64 autograd:           CHAIN_TOL = 1e-4
  * dense chain configurations (default / unfused BN backward / SIMT) against each other: CROSS_TOL = 1e-5
Measured maxima on one NVIDIA B200 (1000 W power limit): products 4.2e-6 (tc_gemm, K=512), 2.0e-6 (dX),
6.1e-7 (dW up to 4737 rows); mean/scale/shift/running mean <= 1e-5; var 1.0e-5 and running var 9.0e-6;
s1|s2 1.7e-5; segmax_bn_bwd and the dY side store <= 1e-5; dW at 1.3 M rows 7.6e-5; chain against float64
1.9e-5.  Where a bound exceeds the 1e-5 target, the reason is float32 accumulation, not the statistics:
  * var: with the cancellation-prone input (|mean| up to ~300, variance ~1) every C element carries the
    rounding of a float32 accumulator of magnitude ~300 (ulp 3e-5); its covariance with C is 1e-5 of the
    variance at 1151 rows.
  * s1|s2: the sums of the layer below add ~1e5 rows of dX whose accumulator rounding does not cancel the
    way the random-sign terms of s1 do (1.7e-5 at 94757 rows, K=256).
  * dW at 1.3 M rows: a CTA accumulates its whole slab (~8800 points) in one float32 tensor-memory
    accumulator before the 148 partials are merged; the error grows with the slab (6e-7 at 4737 rows,
    ~9e-6 at 131072 in the chain test, 7.6e-5 at 1.3 M).
Single-pass TF32 misses PROD_TOL, STAT_TOL and VAR_TOL by at least 10x and S12_TOL by at least 9x at these
shapes and inputs (test_bounds_reject_single_pass_tf32, emulated on the CPU), so a lost lo-term of the
3xTF32 split fails the suite; DW_BIG_TOL is only ~3x below it, the dW cases up to 4737 rows carry that check
for tc_dw.
"""
import copy
import gc

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import nets_ref  # noqa: E402  (checker only)
from test_bf16 import BF16_TOL  # noqa: E402
from test_gpu_parity import close  # noqa: E402

gpu = pytest.mark.gpu

PROD_TOL = 2e-5
STAT_TOL = 1e-5
VAR_TOL = 2e-5
S12_TOL = 2e-5
DW_BIG_TOL = 1e-4
CHAIN_TOL = 1e-4
CROSS_TOL = 1e-5
EPS = 1e-5
MOM = 0.1

# ------------------------------------------------------------------ tc_gemm2.cu configurations
# pick_ns / stages_for of tc_gemm2.cu: a CTA keeps the hi|lo weight slice [NS, K] resident in shared memory
# next to an A ring of 2..4 stages of 32 KB (227 KB per CTA, 1 KB static).  Slices = N / NS.
#
#   N    K    | NS   slices  A-ring stages
#   32   32   | 32   1       4
#   64   64   | 64   1       4
#   128  64   | 128  1       4
#   128  96   | 128  1       3   (ring depth not a power of two)
#   128  128  | 128  1       2
#   128  256  | 64   2       2
#   256  128  | 128  2       2
#   256  256  | 64   4       2
#   64   512  | 32   2       2
# (N=96, K=48) and (N=128, K=512) are unsupported.
FWD_CONFIGS = [(32, 32, 32, 1, 4), (64, 64, 64, 1, 4), (128, 64, 128, 1, 4), (128, 96, 128, 1, 3),
               (128, 128, 128, 1, 2), (128, 256, 64, 2, 2), (256, 128, 128, 2, 2), (256, 256, 64, 4, 2),
               (64, 512, 32, 2, 2)]
# row counts: the dispatch threshold, M % 128 in {1, 127} with fewer tiles than CTAs (epilogue warp quarters
# without rows), and 5 * 148 * 128 + 37 (every CTA walks many tiles: ring and accumulator parities wrap)
FWD_ROWS = [512, 5 * 128 + 1, 8 * 128 + 127, 5 * 148 * 128 + 37]
BIG_ROWS = 1299277  # ~1.3 M rows: the point count of a training batch
DW_ROWS = [32, 33, 2049, 148 * 32 + 1, BIG_ROWS]  # 148*32+1: about half the CTAs get no chunk
DW_SHAPES = [(co, ci) for co in (64, 128, 256) for ci in (32, 64, 128)]


def _fixed_smem(ns, k):
    return (k // 32) * 2 * ns * 32 * 4 + (4 * k + ns + 4 * ns + 4 * ns * 4) * 4 + 4 * 32 * 36 * 4


def _stages(ns, k):
    return min(4, (232448 - 1024 - _fixed_smem(ns, k)) // (2 * 128 * 32 * 4))


def _pick_ns(n, k):
    for ns in (128, 64, 32):
        if n % ns == 0 and (ns != 32 or n <= 64) and _stages(ns, k) >= 2:
            return ns
    return 0


def test_gemm_shapes_reach_every_configuration():
    """The shape table above is what tc_gemm2.cu's slice/ring formula gives (transcribed here); if the kernel's
    shared-memory budget changes, the shapes have to be re-chosen."""
    for n, k, ns, slices, stages in FWD_CONFIGS:
        assert (_pick_ns(n, k), n // _pick_ns(n, k), _stages(_pick_ns(n, k), k)) == (ns, slices, stages), (n, k)
    assert {(ns, stages) for _, _, ns, _, stages in FWD_CONFIGS} >= {(128, 4), (128, 3), (128, 2), (64, 2),
                                                                      (32, 2)}
    assert _pick_ns(128, 512) == 0


# ------------------------------------------------------------------ helpers
@pytest.fixture(scope="module")
def dev():
    from superpoint_graph_b200 import _lib
    _lib.lib()
    return torch.device("cuda:0")


@pytest.fixture
def nan_outputs(monkeypatch):
    """Every buffer ops allocates with torch.empty starts as NaN (integers: -1), so an output element a
    kernel forgot to write cannot pass as a stale value."""
    from superpoint_graph_b200 import ops

    class _Torch(object):
        def __getattr__(self, name):
            return getattr(torch, name)

        @staticmethod
        def empty(*a, **kw):
            t = torch.empty(*a, **kw)
            return t.fill_(float("nan")) if t.is_floating_point() else t.fill_(-1)

    monkeypatch.setattr(ops, "torch", _Torch())


def rel(got, ref):
    got = torch.as_tensor(got)
    ref = torch.as_tensor(ref).to(got.device).double()
    assert got.shape == ref.shape, (got.shape, ref.shape)
    assert bool(torch.isfinite(got).all()), "non-finite values"
    return float((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def check(name, got, ref, tol):
    e = rel(got, ref)
    print("[tc] %-40s err %.2e (bound %.0e)" % (name, e, tol))
    assert e <= tol, "%s: %.3e > %.0e" % (name, e, tol)


def randn(*shape, dev, seed, scale=1.0, offset=0.0):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    return torch.randn(*shape, generator=g, device=dev) * scale + offset


def rand(*shape, dev, seed, lo=0.0, hi=1.0):
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    return torch.rand(*shape, generator=g, device=dev) * (hi - lo) + lo


def affine64(x, scale, shift, relu):
    """float64 value of the prologue relu(fmaf(x, scale, shift)) on float32 operands."""
    x = x.double()
    if scale is not None:
        x = x * scale.double()
    if shift is not None:
        x = x + shift.double()
    return x.clamp_min(0.0) if relu else x


def mask64(y, scale, shift):
    """fmaf(y, scale, shift) > 0 as the kernels evaluate it (the float64 product of two float32 values is exact
    and the sum keeps the sign of the float32 result)."""
    return ((y.double() * scale.double() + shift.double()) > 0).double()


def bn_inputs(y, dev, seed, affine=True):
    """Batch statistics of y (float64, stored as float32) and the fold scale/shift the training forward hands
    to the backward."""
    mu, var = y.double().mean(0), y.double().var(0, unbiased=False)
    C = y.shape[1]
    gamma = rand(C, dev=dev, seed=seed, lo=0.5, hi=1.5) if affine else None
    beta = randn(C, dev=dev, seed=seed + 1, scale=0.3) if affine else None
    sc = (1.0 if gamma is None else gamma.double()) / torch.sqrt(var + EPS)
    sh = (0.0 if beta is None else beta.double()) - mu * sc
    return mu.float(), var.float(), sc.float(), sh.float(), gamma, beta


# ------------------------------------------------------------------ ops.tc_gemm, forward (PRO_AFFINE)
@gpu
@pytest.mark.parametrize("M", FWD_ROWS)
@pytest.mark.parametrize("N,K,ns,slices,stages", FWD_CONFIGS)
def test_tc_gemm_forward_configurations(dev, nan_outputs, N, K, ns, slices, stages, M):
    """Every slice width / ring depth at every row-count edge, with the full prologue and a bias."""
    from superpoint_graph_b200 import ops
    assert ops.tc_supported(M, N, K, K, N)
    A = randn(M, K, dev=dev, seed=1)
    W = randn(N, K, dev=dev, seed=2, scale=K ** -0.5)
    b = randn(N, dev=dev, seed=3)
    sc, sh = rand(K, dev=dev, seed=4, lo=0.5, hi=1.5), randn(K, dev=dev, seed=5)
    C = ops.tc_gemm(A, K, W, K, False, M, N, K, bias=b, a_aff=(sc, sh, True))
    ref = affine64(A, sc, sh, True) @ W.double().t() + b.double()
    check("fwd N=%d K=%d M=%d" % (N, K, M), C, ref, PROD_TOL)


@gpu
def test_tc_gemm_unsupported_shapes(dev):
    from superpoint_graph_b200 import ops
    assert not ops.tc_supported(4096, 96, 48, 48, 96)
    assert not ops.tc_supported(4096, 128, 512, 512, 128)
    assert not ops.tc_supported(511, 128, 128, 128, 128)  # below the dispatch threshold


@gpu
@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("pro", ["none", "scale", "shift", "relu", "all"])
@pytest.mark.parametrize("N,K,M", [(128, 96, 8 * 128 + 127), (256, 256, 5 * 148 * 128 + 37)])
def test_tc_gemm_prologue_combinations(dev, nan_outputs, N, K, M, pro, bias):
    from superpoint_graph_b200 import ops
    A = randn(M, K, dev=dev, seed=11)
    W = randn(N, K, dev=dev, seed=12, scale=K ** -0.5)
    b = randn(N, dev=dev, seed=13) if bias else None
    sc = rand(K, dev=dev, seed=14, lo=0.5, hi=1.5) if pro in ("scale", "all") else None
    sh = randn(K, dev=dev, seed=15) if pro in ("shift", "all") else None
    relu = pro in ("relu", "all")
    aff = None if pro == "none" else (sc, sh, relu)
    C = ops.tc_gemm(A, K, W, K, False, M, N, K, bias=b, a_aff=aff)
    ref = affine64(A, sc, sh, relu) @ W.double().t() + (0.0 if b is None else b.double())
    check("prologue %s bias=%d N=%d K=%d" % (pro, bias, N, K), C, ref, PROD_TOL)


@gpu
@pytest.mark.parametrize("N,K,M", [(64, 64, 5 * 128 + 1), (256, 128, 5 * 148 * 128 + 37), (64, 512, 512)])
def test_tc_gemm_wide_rows_padding_never_read(dev, nan_outputs, N, K, M):
    """lda > K: the padding columns hold NaN; one read of them would poison the row."""
    from superpoint_graph_b200 import ops
    lda = K + 8
    A = randn(M, lda, dev=dev, seed=21)
    A[:, K:] = float("nan")
    W = randn(N, K, dev=dev, seed=22, scale=K ** -0.5)
    sc, sh = rand(K, dev=dev, seed=23, lo=0.5, hi=1.5), randn(K, dev=dev, seed=24)
    C = ops.tc_gemm(A, lda, W, K, False, M, N, K, a_aff=(sc, sh, True))
    check("lda=%d N=%d K=%d M=%d" % (lda, N, K, M), C, affine64(A[:, :K], sc, sh, True) @ W.double().t(), PROD_TOL)


@gpu
@pytest.mark.parametrize("M", [5 * 128 + 1, 5 * 148 * 128 + 37])
@pytest.mark.parametrize("N", [64, 128])
def test_tc_gemm_k_valid(dev, nan_outputs, N, M):
    """First point-wise layer: 14 input features zero-padded to K = 32; the weight image is zero beyond
    k_valid, the weights are read with their own leading dimension (14)."""
    from superpoint_graph_b200 import ops
    A = torch.zeros(M, 32, device=dev)
    A[:, :14] = randn(M, 14, dev=dev, seed=31)
    W = randn(N, 14, dev=dev, seed=32, scale=0.3)
    b = randn(N, dev=dev, seed=33)
    C = ops.tc_gemm(A, 32, W, 14, False, M, N, 32, bias=b, k_valid=14)
    check("k_valid=14 N=%d M=%d" % (N, M), C, A[:, :14].double() @ W.double().t() + b.double(), PROD_TOL)


@gpu
@pytest.mark.parametrize("M", [512, 5 * 148 * 128 + 37])
@pytest.mark.parametrize("Nout,Kin", [(32, 64), (64, 128), (128, 256), (256, 128), (64, 256)])
def test_tc_gemm_transposed_weights(dev, nan_outputs, Nout, Kin, M):
    """Data-gradient form: C[M, Nout] = A[M, Kin] W[Kin, Nout] from the transposed weight image."""
    from superpoint_graph_b200 import ops
    A = randn(M, Kin, dev=dev, seed=41)
    W = randn(Kin, Nout, dev=dev, seed=42, scale=Kin ** -0.5)
    C = ops.tc_gemm(A, Kin, W, Nout, True, M, Nout, Kin)
    check("transposed Nout=%d Kin=%d M=%d" % (Nout, Kin, M), C, A.double() @ W.double(), PROD_TOL)


# ------------------------------------------------------------------ stats=True (+ fold): EPI_STATS
def stats_inputs(M, N, K, dev, seed):
    """Cancellation-prone: A ~ N(100, 1) gives columns of C with |mean| up to a few hundred and variance ~1."""
    A = randn(M, K, dev=dev, seed=seed, offset=100.0)
    W = randn(N, K, dev=dev, seed=seed + 1, scale=K ** -0.5)
    rm0 = randn(N, dev=dev, seed=seed + 2, scale=0.01)
    rv0 = rand(N, dev=dev, seed=seed + 3, lo=0.0, hi=0.01)
    return A, W, rm0, rv0


@gpu
@pytest.mark.parametrize("affine", [True, False])
@pytest.mark.parametrize("N,K,M", [(32, 32, 512), (64, 64, 5 * 128 + 1), (128, 96, 8 * 128 + 127),
                                   (128, 256, 5 * 148 * 128 + 37), (256, 128, 5 * 148 * 128 + 37),
                                   (256, 256, 8 * 128 + 127)])
def test_tc_gemm_stats_and_fold(dev, nan_outputs, N, K, M, affine):
    """Batch statistics, BatchNorm fold and running statistics out of the GEMM's epilogue + merge.  gamma/beta
    None is BatchNorm(affine=False); the running variance takes the unbiased M/(M-1) estimate (2e-4 of it at
    M=512: visible at 1e-5); num_batches_tracked goes up by exactly one."""
    from superpoint_graph_b200 import ops
    A, W, rm0, rv0 = stats_inputs(M, N, K, dev, 51)
    gamma = rand(N, dev=dev, seed=55, lo=0.5, hi=1.5) if affine else None
    beta = randn(N, dev=dev, seed=56, scale=0.3) if affine else None
    rm, rv = rm0.clone(), rv0.clone()
    nbt = torch.full((), 7, dtype=torch.int64, device=dev)
    y, mean, var, scale, shift = ops.tc_gemm(A, K, W, K, False, M, N, K, stats=True,
                                             fold=(gamma, beta, EPS, rm, rv, nbt, MOM))
    y_only, mean2, var2 = ops.tc_gemm(A, K, W, K, False, M, N, K, stats=True)
    ref = A.double() @ W.double().t()
    mu, v = ref.mean(0), ref.var(0, unbiased=False)
    sc = (1.0 if gamma is None else gamma.double()) / torch.sqrt(v + EPS)
    sh = (0.0 if beta is None else beta.double()) - mu * sc
    tag = "N=%d K=%d M=%d affine=%d" % (N, K, M, affine)
    check("stats y " + tag, y, ref, PROD_TOL)
    check("stats mean " + tag, mean, mu, STAT_TOL)
    check("stats var " + tag, var, v, VAR_TOL)
    check("stats scale " + tag, scale, sc, STAT_TOL)
    check("stats shift " + tag, shift, sh, STAT_TOL)
    check("stats running_mean " + tag, rm, (1 - MOM) * rm0.double() + MOM * mu, STAT_TOL)
    check("stats running_var " + tag, rv, (1 - MOM) * rv0.double() + MOM * v * M / (M - 1), VAR_TOL)
    assert int(nbt) == 8
    assert torch.equal(y_only, y) and torch.equal(mean2, mean) and torch.equal(var2, var)


# ------------------------------------------------------------------ PRO_BNBWD (+ EPI_BNRED) and EPI_BNRED alone
def bnbwd_case(M, N, K2, relu, dev, seed):
    """The data gradient of a Conv+BN(+ReLU) layer: G = dL/d(activation) [M, N], raw output y [M, N],
    weight Wd [N, K2]; the layer below has raw output y2 [M, K2]."""
    G = randn(M, N, dev=dev, seed=seed)
    y = randn(M, N, dev=dev, seed=seed + 1, scale=2.0, offset=0.5)
    mu, var, sc, sh, _, _ = bn_inputs(y, dev, seed + 2)
    m = mask64(y, sc, sh) if relu else 1.0
    rstd = 1.0 / torch.sqrt(var.double() + EPS)
    xhat = (y.double() - mu.double()) * rstd
    gz = G.double() * m
    s12 = torch.cat([gz.sum(0), (gz * xhat).sum(0)]).float()
    dY = sc.double() * (gz - s12[:N].double() / M - xhat * s12[N:].double() / M)
    Wd = randn(N, K2, dev=dev, seed=seed + 4, scale=N ** -0.5)
    return G, y, (mu, var, sc, sh, s12), dY, Wd


def bnred_ref(dX, y2, sc2, sh2, mu2, var2, relu2):
    m = mask64(y2, sc2, sh2) if relu2 else 1.0
    gz = dX * m
    xh = (y2.double() - mu2.double()) / torch.sqrt(var2.double() + EPS)
    return gz.sum(0), (gz * xh).sum(0)


BNBWD_SHAPES = [(64, 32, 5 * 128 + 1), (128, 64, 5 * 148 * 128 + 37), (128, 256, 8 * 128 + 127),
                (256, 128, 512), (256, 256, 5 * 148 * 128 + 37)]  # (layer cout N, layer cin K2, M)


@gpu
@pytest.mark.parametrize("want_dy", [True, False])
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("N,K2,M", BNBWD_SHAPES)
def test_tc_gemm_bnbwd_prologue_and_bnred(dev, nan_outputs, N, K2, M, relu, want_dy):
    """BatchNorm(+ReLU) backward in the prologue, optional dY side store (slice 0 only: with 2 and 4 slices
    every other slice must leave it alone, and every row must still be written), BatchNorm-backward sums of
    the layer below in the epilogue.  The layer below has a ReLU: without one its s1 = sum_m dX is
    analytically zero (sum_m dY = 0 after a batch-statistics BatchNorm) and holds only rounding noise."""
    from superpoint_graph_b200 import ops
    G, y, (mu, var, sc, sh, s12), dY_ref, Wd = bnbwd_case(M, N, K2, relu, dev, 61)
    y2 = randn(M, K2, dev=dev, seed=66, offset=0.2)
    mu2, var2, sc2, sh2, _, _ = bn_inputs(y2, dev, 67)
    res = ops.tc_gemm(G, N, Wd, K2, True, M, K2, N, bnbwd=(y, N, sc, sh, relu, mu, var, s12, EPS, want_dy),
                      bnred=(y2, K2, sc2, sh2, mu2, var2, EPS, True))
    dX, rest = res[0], list(res[1:])
    dX_ref = dY_ref @ Wd.double()
    tag = "N=%d K2=%d M=%d relu=%d" % (N, K2, M, relu)
    check("bnbwd dX " + tag, dX, dX_ref, PROD_TOL)
    if want_dy:
        check("bnbwd dY side store " + tag, rest.pop(0), dY_ref, STAT_TOL)
    s12b = rest.pop(0)
    r1, r2 = bnred_ref(dX_ref, y2, sc2, sh2, mu2, var2, True)
    check("bnred s1 " + tag, s12b[:K2], r1, S12_TOL)
    check("bnred s2 " + tag, s12b[K2:], r2, S12_TOL)
    assert not rest


@gpu
@pytest.mark.parametrize("affine", [True, False])
@pytest.mark.parametrize("e_relu", [True, False])
@pytest.mark.parametrize("N,K,M", [(64, 128, 5 * 128 + 1), (256, 64, 5 * 148 * 128 + 37), (128, 256, 512)])
def test_tc_gemm_bnred_epilogue(dev, nan_outputs, N, K, M, e_relu, affine):
    """EPI_BNRED behind a plain (transposed-weight) GEMM; e_scale/e_shift None is a BatchNorm without affine
    parameters whose fold the caller did not materialise (scale 1, shift 0 in the mask)."""
    from superpoint_graph_b200 import ops
    A = randn(M, K, dev=dev, seed=71)
    W = randn(K, N, dev=dev, seed=72, scale=K ** -0.5)
    y2 = randn(M, N, dev=dev, seed=73, offset=0.2)
    mu2, var2, sc2, sh2, _, _ = bn_inputs(y2, dev, 74)
    if not affine:
        sc2 = sh2 = None
    C, s12 = ops.tc_gemm(A, K, W, N, True, M, N, K, bnred=(y2, N, sc2, sh2, mu2, var2, EPS, e_relu))
    C_ref = A.double() @ W.double()
    ones, zeros = torch.ones(N, device=dev), torch.zeros(N, device=dev)
    r1, r2 = bnred_ref(C_ref, y2, ones if sc2 is None else sc2, zeros if sh2 is None else sh2, mu2, var2, e_relu)
    tag = "N=%d K=%d M=%d relu=%d affine=%d" % (N, K, M, e_relu, affine)
    check("bnred C " + tag, C, C_ref, PROD_TOL)
    check("bnred s1 " + tag, s12[:N], r1, S12_TOL)
    check("bnred s2 " + tag, s12[N:], r2, S12_TOL)


# ------------------------------------------------------------------ ops.tc_dw
@gpu
@pytest.mark.parametrize("M", DW_ROWS)
@pytest.mark.parametrize("co,ci", DW_SHAPES)
def test_tc_dw_shapes_and_rows(dev, nan_outputs, co, ci, M):
    """All nine instantiations (co=64 runs the zero-padded 128-row accumulator) at every chunk edge; leading
    dimensions wider than co/ci with NaN padding; the input prologue of the layer below."""
    from superpoint_graph_b200 import ops
    lddy, ldp = co + 8, ci + 4
    dY = randn(M, lddy, dev=dev, seed=81)
    P = randn(M, ldp, dev=dev, seed=82)
    dY[:, co:] = float("nan")
    P[:, ci:] = float("nan")
    sc, sh = rand(ci, dev=dev, seed=83, lo=0.5, hi=1.5), randn(ci, dev=dev, seed=84)
    dW = ops.tc_dw(dY, lddy, P, ldp, M, co, ci, p_aff=(sc, sh, True))
    ref = dY[:, :co].double().t() @ affine64(P[:, :ci], sc, sh, True)
    check("dW co=%d ci=%d M=%d" % (co, ci, M), dW, ref, DW_BIG_TOL if M == BIG_ROWS else PROD_TOL)


@gpu
@pytest.mark.parametrize("pro", ["none", "scale", "shift", "relu", "scale+shift"])
@pytest.mark.parametrize("co,ci,M", [(64, 128, 2049), (256, 32, 148 * 32 + 1), (128, 64, BIG_ROWS)])
def test_tc_dw_prologue_combinations(dev, nan_outputs, co, ci, M, pro):
    from superpoint_graph_b200 import ops
    dY = randn(M, co, dev=dev, seed=91)
    P = randn(M, ci, dev=dev, seed=92)
    sc = rand(ci, dev=dev, seed=93, lo=0.5, hi=1.5) if "scale" in pro else None
    sh = randn(ci, dev=dev, seed=94) if "shift" in pro else None
    relu = pro == "relu"
    aff = None if pro == "none" else (sc, sh, relu)
    dW = ops.tc_dw(dY, co, P, ci, M, co, ci, p_aff=aff)
    check("dW %s co=%d ci=%d M=%d" % (pro, co, ci, M), dW, dY.double().t() @ affine64(P, sc, sh, relu),
          DW_BIG_TOL if M == BIG_ROWS else PROD_TOL)


# ------------------------------------------------------------------ packing (tc_pack.cu)
@gpu
def test_weight_packers_are_bit_identical(dev):
    """The batched prepack table, the on-demand packer (the one every GEMM test above validates) and the
    scaled packer with row_scale=None give the same bits, incl. transposed images, k_valid < K and a weight
    leading dimension wider than the row."""
    from superpoint_graph_b200 import _lib, ops
    W14 = randn(64, 14, dev=dev, seed=101)
    W2 = randn(128, 64, dev=dev, seed=102)
    Wwide = randn(256, 136, dev=dev, seed=103)  # ldw 136, 128 valid columns
    Wt14 = randn(14, 64, dev=dev, seed=104)     # transposed with k_valid=14 rows
    jobs = [(W14, 14, False, 64, 32, 14), (W2, 64, False, 128, 64, 64), (W2, 64, True, 64, 128, 128),
            (Wwide, 136, False, 256, 128, 128), (Wwide, 136, True, 128, 256, 256), (Wt14, 64, True, 64, 32, 14)]
    ops.PACK_CACHE.clear()
    try:
        ops.prepack(jobs)
        batched = dict(ops.PACK_CACHE)
        ops.PACK_CACHE.clear()
        for (W, ldw, tr, N, K, kv) in jobs:
            key = (W.data_ptr(), ldw, int(tr), N, K, kv)
            on_demand = ops._weight_image(W, ldw, tr, N, K, kv, dev)
            assert torch.equal(on_demand.view(torch.int32), batched[key].view(torch.int32)), key
            if not tr:
                scaled = torch.full((2 * N * K,), float("nan"), device=dev)
                _lib.call("spg_tc_pack_weights_scaled", W, ldw, None, N, K, kv, scaled, _lib.current_stream())
                assert torch.equal(scaled.view(torch.int32), on_demand.view(torch.int32)), key
    finally:
        ops.PACK_CACHE.clear()  # keyed by address: nothing of this test may outlive it


# ------------------------------------------------------------------ determinism
@gpu
def test_fused_reductions_and_dw_are_deterministic(dev):
    """The merges fold the per-CTA partials in a fixed order: identical calls give identical bits."""
    from superpoint_graph_b200 import ops
    M = 5 * 148 * 128 + 37
    A, W, rm0, rv0 = stats_inputs(M, 128, 128, dev, 111)
    gamma, beta = rand(128, dev=dev, seed=115, lo=0.5, hi=1.5), randn(128, dev=dev, seed=116)
    runs = []
    for _ in range(2):
        rm, rv = rm0.clone(), rv0.clone()
        nbt = torch.zeros((), dtype=torch.int64, device=dev)
        out = ops.tc_gemm(A, 128, W, 128, False, M, 128, 128, stats=True,
                          fold=(gamma, beta, EPS, rm, rv, nbt, MOM))
        runs.append([t.clone() for t in out] + [rm, rv])
    G, y, (mu, var, sc, sh, s12), _, Wd = bnbwd_case(M, 256, 128, True, dev, 117)
    y2 = randn(M, 128, dev=dev, seed=118)
    mu2, var2, sc2, sh2, _, _ = bn_inputs(y2, dev, 119)
    bw = [[t.clone() for t in ops.tc_gemm(G, 256, Wd, 128, True, M, 128, 256,
                                          bnbwd=(y, 256, sc, sh, True, mu, var, s12, EPS, True),
                                          bnred=(y2, 128, sc2, sh2, mu2, var2, EPS, True))] for _ in range(2)]
    dYb = randn(BIG_ROWS, 256, dev=dev, seed=120)
    Pb = randn(BIG_ROWS, 128, dev=dev, seed=121)
    dw = [ops.tc_dw(dYb, 256, Pb, 128, BIG_ROWS, 256, 128).clone() for _ in range(2)]
    for a, b in zip(runs[0] + bw[0] + dw[:1], runs[1] + bw[1] + dw[1:]):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


# ------------------------------------------------------------------ ops.segmax_bn_bwd
@gpu
@pytest.mark.parametrize("B,L,C,relu", [(601, 128, 64, True), (301, 128, 256, True), (1000, 20, 128, False),
                                        (3, 128, 32, True)])
def test_segmax_bn_bwd_vs_float64_autograd(dev, nan_outputs, B, L, C, relu):
    """Max-pool backward fused with the BatchNorm(+ReLU) backward, with the kernel's own argmax, against float64
    autograd of relu(bn(Y)) followed by the gather at that argmax (BatchNorm with batch statistics; the ReLU
    mask is the kernel's float32 one)."""
    from superpoint_graph_b200 import ops
    Y = randn(B * L, C, dev=dev, seed=131, scale=1.5, offset=0.3)
    mu, var, sc, sh, gamma, beta = bn_inputs(Y, dev, 132)
    pooled = torch.empty(B, C, device=dev)
    argmax = ops.segmax_fwd(Y, C, B, L, C, sc, sh, relu, pooled, C)
    gp = randn(B, C, dev=dev, seed=134)
    s1, s2, dY = ops.segmax_bn_bwd(gp, C, argmax, Y, C, sc, sh, mu, var, EPS, relu, B, L, C)
    Yr = Y.double().requires_grad_(True)
    g64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    xhat = (Yr - Yr.mean(0)) / torch.sqrt(Yr.var(0, unbiased=False) + EPS)
    act = (xhat * g64 + b64) * (mask64(Y, sc, sh) if relu else 1.0)
    act.view(B, L, C).gather(1, argmax.long().view(B, 1, C)).backward(gp.double().view(B, 1, C))
    tag = "B=%d L=%d C=%d relu=%d" % (B, L, C, relu)
    check("segmax_bn_bwd s1 " + tag, s1, b64.grad, STAT_TOL)
    check("segmax_bn_bwd s2 " + tag, s2, g64.grad, STAT_TOL)
    check("segmax_bn_bwd dY " + tag, dY, Yr.grad, STAT_TOL)


# ------------------------------------------------------------------ single-pass TF32 would fail the bounds
def _tf32(x):
    """float32 -> float64 value of to_tf32(x): 10-bit mantissa, rounded half away from zero."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x1000)) & np.uint32(0xffffe000)).view(np.float32).astype(np.float64)


def _rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def test_bounds_reject_single_pass_tf32():
    """Emulates single-pass TF32 (both operands rounded to tf32, exact float64 accumulation) at the (N, K) and
    (co, ci) shapes and with the input distributions of the tests above, and requires every bound to be at
    least 10x below the error that gives.  Rows are capped at 16384: the relative error of a sum of
    random-sign terms, and the per-column bias that rounding the weights causes, do not depend on the row
    count."""
    rng = np.random.default_rng(0)
    M = 16384
    worst = {}

    def note(name, e):
        worst[name] = min(worst.get(name, np.inf), e)

    for N, K, _, _, _ in FWD_CONFIGS:
        A = rng.standard_normal((M, K)).astype(np.float32)
        W = (rng.standard_normal((N, K)) * K ** -0.5).astype(np.float32)
        note("product", _rel(_tf32(A) @ _tf32(W).T, A.astype(np.float64) @ W.astype(np.float64).T))
        # statistics inputs: A ~ N(100, 1)
        A = (100 + rng.standard_normal((M, K))).astype(np.float32)
        exact, one = A.astype(np.float64) @ W.astype(np.float64).T, _tf32(A) @ _tf32(W).T
        mu, mu1 = exact.mean(0), one.mean(0)
        v, v1 = exact.var(0), one.var(0)
        g = rng.uniform(0.5, 1.5, N)
        sc, sc1 = g / np.sqrt(v + EPS), g / np.sqrt(v1 + EPS)
        note("mean", _rel(mu1, mu))
        note("var", _rel(v1, v))
        note("scale", _rel(sc1, sc))
        note("shift", _rel(-mu1 * sc1, -mu * sc))
        rm0, rv0 = rng.standard_normal(N) * 0.01, rng.uniform(0, 0.01, N)
        note("running_mean", _rel((1 - MOM) * rm0 + MOM * mu1, (1 - MOM) * rm0 + MOM * mu))
        note("running_var", _rel((1 - MOM) * rv0 + MOM * v1, (1 - MOM) * rv0 + MOM * v))
    for co, ci in DW_SHAPES:
        dY = rng.standard_normal((M, co)).astype(np.float32)
        P = rng.standard_normal((M, ci)).astype(np.float32)
        note("dW", _rel(_tf32(dY).T @ _tf32(P), dY.astype(np.float64).T @ P.astype(np.float64)))
    for N, K2, _ in BNBWD_SHAPES:  # s1|s2 of the layer below from a single-pass dX
        dY = rng.standard_normal((M, N)).astype(np.float32)
        Wd = (rng.standard_normal((N, K2)) * N ** -0.5).astype(np.float32)
        exact, one = dY.astype(np.float64) @ Wd.astype(np.float64), _tf32(dY) @ _tf32(Wd)
        y2 = rng.standard_normal((M, K2)) + 0.2
        m = (y2 > 0).astype(np.float64)
        xh = (y2 - y2.mean(0)) / y2.std(0)
        note("s1", _rel((one * m).sum(0), (exact * m).sum(0)))
        note("s2", _rel((one * m * xh).sum(0), (exact * m * xh).sum(0)))
        note("dX", _rel(one, exact))
    bounds = dict(product=PROD_TOL, dX=PROD_TOL, dW=PROD_TOL, mean=STAT_TOL, var=VAR_TOL, scale=STAT_TOL,
                  shift=STAT_TOL, running_mean=STAT_TOL, running_var=VAR_TOL, s1=S12_TOL, s2=S12_TOL)
    for name, tol in bounds.items():
        margin = 9 if name in ("s1", "s2") else 10  # (see the module docstring)
        print("[tf32x1] %-13s smallest error %.2e, bound %.0e" % (name, worst[name], tol))
        assert worst[name] >= margin * tol, (name, worst[name], tol)


# ------------------------------------------------------------------ dense chain, training mode
def _chain_module(seed):
    torch.manual_seed(seed)
    seq = nn.Sequential(nn.Linear(64, 128), nn.BatchNorm1d(128), nn.ReLU(),
                        nn.Linear(128, 256), nn.BatchNorm1d(256), nn.ReLU(),
                        nn.Linear(256, 128), nn.BatchNorm1d(128), nn.ReLU())
    with torch.no_grad():
        for m in seq.modules():
            if isinstance(m, nn.BatchNorm1d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.normal_(0, 0.2)
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    return seq


def _run_chain(seq0, X, GY, dev, monkeypatch, cfg):
    """One training forward + backward of dense.run_sequential; returns its results and the ReLU masks of its
    own float32 pre-activations."""
    from superpoint_graph_b200 import dense, ops
    seq = copy.deepcopy(seq0).to(dev)
    saved = []
    orig = dense.chain_forward

    def recording(inp, M, specs, params, training, sv=None):
        out = orig(inp, M, specs, params, training, sv)
        saved.append(sv)
        return out

    with monkeypatch.context() as mp:
        mp.setattr(dense, "chain_forward", recording)
        if cfg == "unfused_bnbwd":
            mp.setattr(ops, "USE_FUSED_BNBWD", [False])
        elif cfg == "simt":
            mp.setattr(ops, "USE_TC", [False])
        x = X.clone().requires_grad_(True)
        ops.prof_reset()
        y = dense.run_sequential(seq, x, True)
        y.backward(GY)
        torch.cuda.synchronize()
        kernels = ops.prof_collect()
    (sv,) = saved
    masks = [mask64(nxt.raw, nxt.scale, nxt.shift) for _, nxt, _, _ in sv]
    res = {"out": y.detach(), "grad_in": x.grad}
    res.update(("grad " + k, p.grad) for k, p in seq.named_parameters())
    res.update(("buffer " + k, b) for k, b in seq.named_buffers())
    return res, masks, kernels


def _ref_chain(seq0, X, GY, dev, masks):
    """float64 autograd of the same module; each ReLU takes the mask of the float32 run's pre-activation."""
    seq = copy.deepcopy(seq0).double().to(dev)
    relus = [m for m in seq.modules() if isinstance(m, nn.ReLU)]
    for r, m in zip(relus, masks):
        r.register_forward_hook(lambda mod, inp, out, m=m: inp[0] * m)
    x = X.double().requires_grad_(True)
    seq.train()
    y = seq(x)
    y.backward(GY.double())
    res = {"out": y.detach(), "grad_in": x.grad}
    res.update(("grad " + k, p.grad) for k, p in seq.named_parameters())
    res.update(("buffer " + k, b) for k, b in seq.named_buffers())
    return res


PRE_BN_BIASES = ("grad 0.bias", "grad 3.bias", "grad 6.bias")  # analytically zero: BatchNorm removes the mean


@gpu
@pytest.mark.parametrize("M", [511, 512, 2049, 131072])
def test_dense_chain_training_vs_float64(dev, monkeypatch, M):
    """Linear+BatchNorm+ReLU widths 64-128-256-128 through dense.run_sequential in training mode: M=511 runs
    the SIMT GEMMs, 512 the tcgen05 forward with fused statistics and the lazy BNBWD+BNRED data gradients,
    2049 and 131072 also tc_dw.  Three configurations (default, USE_FUSED_BNBWD off, USE_TC off) against a
    float64 copy of the module (CHAIN_TOL) and against each other (CROSS_TOL).  A one-ulp difference of a
    pre-activation near zero can flip a ReLU mask between two float32 runs (20 of 6.7e7 elements between
    the SIMT and the tensor-core forward at 131072 rows, none elsewhere); a flip moves that row's input
    gradient by ~10 % of the tensor's maximum, so gradients are compared across configurations only when
    the masks agree, and flips must stay below 1e-6 of the elements.  Each configuration is always held to
    its own float64 reference.  Biases in front of a BatchNorm have an analytically zero gradient: the
    chain returns exact zeros."""
    seq0 = _chain_module(M)
    X = randn(M, 64, dev=dev, seed=141)
    GY = randn(M, 128, dev=dev, seed=142)
    runs = {}
    for cfg in ("default", "unfused_bnbwd", "simt"):
        got, masks, kernels = _run_chain(seq0, X, GY, dev, monkeypatch, cfg)
        tc, dw = kernels.get("tc_gemm_3xtf32", (0, 0))[0], kernels.get("tc_dw_3xtf32", (0, 0))[0]
        assert (tc > 0) == (M >= 512 and cfg != "simt") and (dw > 0) == (M >= 2048 and cfg != "simt"), kernels
        want = _ref_chain(seq0, X, GY, dev, masks)
        scale = max(float(want[k].abs().max()) for k in want if k.startswith("grad "))
        for k, w in want.items():
            if k in PRE_BN_BIASES:
                assert not bool(got[k].any()) and float(w.abs().max()) <= 1e-9 * scale, k
            elif k.endswith("num_batches_tracked"):
                assert int(got[k]) == int(w) == 1
            else:
                check("chain M=%d %s %s" % (M, cfg, k), got[k], w, CHAIN_TOL)
        runs[cfg] = (got, masks)
    base, base_masks = runs["default"]
    for cfg in ("unfused_bnbwd", "simt"):
        got, masks = runs[cfg]
        flips = sum(int((a != b).sum()) for a, b in zip(masks, base_masks))
        print("[tc] chain M=%d %s: %d ReLU mask differences against the default run" % (M, cfg, flips))
        assert flips <= 1e-6 * sum(m.numel() for m in masks)
        for k, w in base.items():
            if k in PRE_BN_BIASES or k.endswith("num_batches_tracked") or (flips and k.startswith("grad")):
                continue
            check("chain M=%d %s vs default %s" % (M, cfg, k), got[k], w, CROSS_TOL)


# ------------------------------------------------------------------ eval after training (folded weight images)
def _small_trainer(dev, seed, dtype="f32"):
    from superpoint_graph_b200.trainer import Trainer, create_model, make_args
    args = make_args(model_config="gru_3_1_1_1_0,f_13")
    torch.manual_seed(seed)
    model = create_model(args).to(dev)
    return Trainer(model, args, dtype=dtype), args


def _oracle_logits(tr, args, batch):
    from superpoint_graph_b200 import workloads
    pcfg, mcfg = workloads.oracle_cfg(args)
    sd_ptn = {k: v.detach().cpu().clone() for k, v in tr.model.ptn.state_dict().items()}
    sd_ecc = {k: v.detach().cpu().clone() for k, v in tr.model.ecc.state_dict().items()}
    with torch.no_grad():
        return nets_ref.spg_forward(batch, sd_ptn, sd_ecc, pcfg, mcfg, False)


def _eval(tr, db, dtype):
    """Trainer.eval_step in the given trunk arithmetic (the Trainer reads its dtype on every call)."""
    from superpoint_graph_b200 import ops
    saved, tr.dtype = tr.dtype, dtype
    try:
        ops.prof_reset()
        out = tr.eval_step(db).clone()
        assert any(k.startswith("pointnet_fused_eval") for k in ops.prof_collect())  # the cached-image path
        return out
    finally:
        tr.dtype = saved


@gpu
@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_eval_after_training_steps_uses_the_new_weights(dev, dtype):
    """eval_step, two train_steps, eval_step (validation between epochs): the second evaluation must run the
    trained parameters and running statistics, not the folded image cached by the first."""
    from superpoint_graph_b200.synthetic import make_batch
    from superpoint_graph_b200.trainer import HostBatch
    tr, args = _small_trainer(dev, 5)
    batch = make_batch(n_nodes=200, seed=11)
    db = HostBatch(batch).to_device(dev)
    before = _eval(tr, db, dtype)
    tr.train_step(db)
    tr.train_step(db)
    after = _eval(tr, db, dtype)
    want = _oracle_logits(tr, args, batch)
    err = rel(after.cpu(), want)
    print("[tc] eval after training (%s): err %.2e vs oracle; before-training logits differ by %.2e"
          % (dtype, err, rel(before.cpu(), want)))
    assert err <= (1e-4 if dtype == "f32" else BF16_TOL), err


@gpu
def test_replay_eval_refuses_a_graph_captured_before_an_update(dev):
    from superpoint_graph_b200.synthetic import make_batch
    from superpoint_graph_b200.trainer import HostBatch
    tr, args = _small_trainer(dev, 6)
    batch = make_batch(n_nodes=200, seed=12)
    db = HostBatch(batch).to_device(dev)
    key = tr.capture_eval(db, key=0)
    tr.replay_eval(key)
    tr.train_step(db)
    with pytest.raises(RuntimeError, match="capture"):
        tr.replay_eval(key)
    eager = tr.eval_step(db).clone()
    key = tr.capture_eval(db, key=0)
    assert torch.equal(tr.replay_eval(key), eager)
    close(eager, _oracle_logits(tr, args, batch))


@gpu
def test_eval_of_a_new_model_after_the_old_one_was_freed(dev):
    """Model B, built after model A (same architecture, other seed) was evaluated and freed, may get A's
    allocator blocks with equal version counts; its eval must still use its own weights."""
    from superpoint_graph_b200.synthetic import make_batch
    from superpoint_graph_b200.trainer import HostBatch
    batch = make_batch(n_nodes=200, seed=13)
    db = HostBatch(batch).to_device(dev)
    ptrs = []
    for seed in (7, 8):
        tr, args = _small_trainer(dev, seed)
        out = tr.eval_step(db).clone()
        close(out, _oracle_logits(tr, args, batch))
        ptrs.append(tr.flat.data_ptr())
        del tr
        gc.collect()
    print("[tc] model B's parameters %s model A's address" % ("reuse" if ptrs[0] == ptrs[1] else "do not reuse"))
