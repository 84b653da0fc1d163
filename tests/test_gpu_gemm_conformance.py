"""The tcgen05 GEMMs of csrc/transform.cu (forward, dgrad, split-K wgrad, fused ReLU + dropout epilogue, the consuming
ranking epilogues) against a float64 product of the bf16 operand planes the kernels read.

The reference is built from the planes themselves (read back after the split), so the GEMM is tested apart from the
splitting, which has its own bitwise test.  In fp32 mode the kernels accumulate ``hi*hi + hi*lo + lo*hi``, in bf16 mode
``hi*hi``; the float64 reference forms the same products.  Two kinds of cases:

* exact: inputs ``h + j * 2^-10`` (h = +-1, j in {-1, 0, 1}) and zeros split into hi = h, lo = j * 2^-10 without
  rounding ties, so every product and partial sum is a multiple of 2^-10 far below 2^14 and the accumulation is exact in
  any order.  Integer bias, dropout scale 2: the kernel must equal the reference bit for bit.  At K >= 1,000 only this
  detects one missing term or one missing lo product.
* random: ``|got - ref| <= (T + 3) * 2^-23 * sum|terms| + 2^-24 * |bias|`` with T the number of product terms per output
  (K or 3K; 2^-23 because the rounding inside the tensor core's adder tree is not documented), carried through the ReLU
  (1-Lipschitz) and the dropout scale plus one rounding.  A difference where the bound is 0, or a NaN, fails.

The worst error-to-bound ratio of each family is printed when the module finishes (``pytest -s``).
"""
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M32 = 0xFFFFFFFF
E23 = 2.0 ** -23
U = 2.0 ** -24
BM, BK, KBN, BNMAX, WG_BK = 128, 64, 128, 256, 32     # tile constants of csrc/transform.cu
MODES = ["fp32", "bf16"]

_WORST = {}


@pytest.fixture(scope="module")
def ops(lib_built):
    from primekg_rgcn_linkprediction_b200 import ops
    return ops


@pytest.fixture(scope="module")
def lib(lib_built):
    from primekg_rgcn_linkprediction_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for fam in sorted(_WORST):
        print(f"\n[gemm conformance] {fam}: worst |err| / bound = {_WORST[fam]:.3g}", end="")
    print()


# ---- host tile choice of transform.cu, replicated ---------------------------------------------------------------------
def _ru(x, g):
    return (x + g - 1) // g * g


def tile_n(N, gran, bn_max=BNMAX):
    """(n_tiles, BN) of transform.cu's tile_n."""
    np_ = _ru(N, gran)
    nt = (np_ + bn_max - 1) // bn_max
    return nt, _ru((np_ + nt - 1) // nt, gran)


def launch_choice(entry, mode, M, K, d_out, xf, sm, wide_tiles=True, wide_fp32=0, narrow_small=True):
    """(SPLIT, B_MN, BNT, XF, BN) of the gemm_kmajor_kernel instantiation the host code launches.  ``entry``: fwd /
    fwd_w / dgrad / dgrad_w; K is the layer's K1 + K2; xf: 0 plain, 1 fused dropout, 2 bf16 copy or scattered rows."""
    wide_bn = 256 if wide_tiles else KBN
    if entry == "fwd":
        _, bn = tile_n(d_out, 32, KBN)
    elif entry == "fwd_w":
        wide = d_out > KBN and (mode == "bf16" or wide_fp32 == 1 or (wide_fp32 == 2 and K <= 256))
        nt, bn = tile_n(d_out, 32, wide_bn if wide else KBN)
        if narrow_small and d_out % 64 == 0 and d_out >= 128 and (M + BM - 1) // BM * nt * 2 <= sm:
            _, bn = tile_n(d_out, 32, 64)
    elif entry == "dgrad":
        _, bn = tile_n(K, 32, KBN)
    else:
        _, bn = tile_n(K, 32, wide_bn if K > KBN else KBN)
    return mode == "fp32", entry == "fwd_w", 256 if bn > 128 else 128, xf, bn


def bn_class(bn):
    """TMEM accumulator width and whether the MN-major B loads whole 64-column chunks."""
    return (32 if bn <= 32 else 64 if bn <= 64 else 128 if bn <= 128 else 256, bn % 64 == 0)


def wgrad_splits(nodes, tiles, sm):
    s = sm // tiles
    s = min(s, (nodes + 4 * WG_BK - 1) // (4 * WG_BK), 64)
    return max(s, 1)


def _sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- operands and references ------------------------------------------------------------------------------------------
def _gen(seed):
    g = torch.Generator(device=DEV)
    g.manual_seed(seed)
    return g


def _exact(shape, g, zero_frac=0.2):
    """h + j * 2^-10 (h = +-1, j in {-1, 0, 1}) with exact zeros: hi = h, lo = j * 2^-10 exactly."""
    h = torch.randint(0, 2, shape, generator=g, device=DEV) * 2 - 1
    j = torch.randint(-1, 2, shape, generator=g, device=DEV)
    x = (h + j * 2.0 ** -10).float()
    return torch.where(torch.rand(shape, generator=g, device=DEV) < zero_frac, 0.0, x)


def _random(shape, g):
    """normal values with row scales over 2^-6 .. 2^6: small outputs must be as right as large ones."""
    x = torch.randn(shape, generator=g, device=DEV)
    return x * torch.exp2(torch.randint(-6, 7, (shape[0], 1), generator=g, device=DEV).float())


def _vals(kind, shape, g):
    """exact or random values; an empty matrix is a view of a one-row allocation (the C ABI wants non-null pointers)."""
    n = shape[0]
    full = (max(n, 1),) + tuple(shape[1:])
    return (_exact(full, g) if kind == "exact" else _random(full, g))[:n]


def _alloc_planes(ops, rows, cols, mode):
    hi, lo = ops.alloc_planes(max(rows, 1), cols, mode, DEV)
    return hi[:rows], (None if lo is None else lo[:rows])


def _bias(kind, n, g):
    if kind == "exact":
        return torch.randint(-3, 4, (n,), generator=g, device=DEV).float()
    return torch.randn(n, generator=g, device=DEV)


def _split_ref(x):
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)


def _planes(ops, mats, mode):
    """fp32 matrices (concatenated along columns) -> bf16 planes, one split_planes call per block (col0 offsets)."""
    n = mats[0].size(0)
    P = _alloc_planes(ops, n, sum(m.size(1) for m in mats), mode)
    c0 = 0
    for m in mats:
        ops.split_planes(m, P, col0=c0)
        c0 += m.size(1)
    return P


def _wplanes(wp, K, N, mode):
    """(hi, lo | None) [K, ld] views of an rgcn_prepare_weights buffer (ld = N rounded up to 8)."""
    ld = _ru(N, 8)
    nbytes = K * ld * 2
    hi = wp[:nbytes].view(torch.bfloat16).view(K, ld)
    off = _ru(nbytes, 1024)
    lo = wp[off:off + nbytes].view(torch.bfloat16).view(K, ld) if mode == "fp32" else None
    return hi, lo


def _prod(Ah, Al, Bh, Bl, mode):
    """float64 (A @ B, sum |terms|, terms per output) from bf16 planes, B as [K, N]."""
    a, b = Ah.double(), Bh.double()
    ref, S = a @ b, a.abs() @ b.abs()
    T = Ah.size(1)
    if mode == "fp32":
        al, bl = Al.double(), Bl.double()
        ref = ref + a @ bl + al @ b
        S = S + a.abs() @ bl.abs() + al.abs() @ b.abs()
        T *= 3
    return ref, S, T


def _check(fam, got, ref, bound, what):
    got = got.double()
    err = (got - ref).abs()
    bad = ~(err <= bound)                                # NaN fails
    pos = bound > 0
    worst = float((err[pos] / bound[pos]).max()) if bool(pos.any()) else 0.0
    _WORST[fam] = max(_WORST.get(fam, 0.0), worst)
    if bool(bad.any()):
        i = int(bad.flatten().nonzero()[0])
        raise AssertionError(f"{fam} {what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at "
                             f"flat index {i}: got {float(got.flatten()[i])!r}, ref {float(ref.flatten()[i])!r}, "
                             f"bound {float(bound.flatten()[i]):.3g}")


def _check_exact(fam, got, ref, what):
    _WORST.setdefault(fam, 0.0)
    bad = got.double() != ref
    if bool(bad.any()):
        i = int(bad.flatten().nonzero()[0])
        raise AssertionError(f"{fam} {what} (exact): {int(bad.sum())} of {bad.numel()} elements differ; first at flat "
                             f"index {i}: got {float(got.flatten()[i])!r}, want {float(ref.flatten()[i])!r}")


def _epilogue_ref(acc, S, T, bias, relu, scale=None, keep=None):
    """(value, bound) of relu(acc + bias) (* scale where kept) in float64."""
    bound = (T + 3) * E23 * S
    v = acc
    if bias is not None:
        b = bias.double()[None, :]
        v = v + b
        bound = bound + U * b.abs()
    if relu:
        v = v.clamp(min=0)
    if keep is not None:
        v = torch.where(keep, v * scale, 0.0)
        bound = torch.where(keep, bound * scale + U * v.abs(), 0.0)
    return v, bound


# ---- the dropout hash of gemm_common.cuh --------------------------------------------------------------------------------
def _pcg(x):
    state = (x * 747796405 + 2891336453) & M32
    word = (((state >> ((state >> 28) + 4)) ^ state) * 277803737) & M32
    return ((word >> 22) ^ word) & M32


def drop_thresh(p):
    return min(max(int(float(np.float32(p)) * 65536.0 + 0.5), 1), 65535)


def drop_scale(p):
    return float(np.float32(1.0) / (np.float32(1.0) - np.float32(p)))


def drop_keep(rows, row_offset, N, p, seed, c, device=DEV):
    """bool [rows, N]: element (row, col) of the call that read counter value c survives the fused dropout."""
    key = (_pcg((seed & M32) ^ (c & M32)) + (c >> 32)) & M32
    r = torch.arange(rows, device=device, dtype=torch.int64)[:, None] + row_offset
    col = torch.arange(N, device=device, dtype=torch.int64)[None, :]
    e4 = r * N + (col & ~3)                              # first element of the aligned group of four
    bk = _pcg((key + (e4 >> 32) * 0x9E3779B9) & M32)
    lo = e4 & M32
    h0, h1 = _pcg(lo ^ bk), _pcg(((lo + 2) & M32) ^ bk)
    sub = col & 3
    bits = torch.where(sub == 0, h0 & 0xFFFF, torch.where(sub == 1, h0 >> 16, torch.where(sub == 2, h1 & 0xFFFF, h1 >> 16)))
    return bits >= drop_thresh(p)


# =========================================================================================================================
# a. rgcn_split_planes / rgcn_prepare_weights
# =========================================================================================================================
@pytest.mark.parametrize("cols", [4, 12, 100, 1024])
@pytest.mark.parametrize("rows", [0, 1, 333])
def test_split_planes_bitwise(ops, lib, rows, cols):
    g = _gen(rows * 7 + cols)
    x = _vals("random", (rows, cols), g)
    mask = torch.randn(max(rows, 1), cols, generator=g, device=DEV)[:rows]
    if rows:
        mask[0, : min(cols, 3)] = float("nan")            # a NaN in the mask zeroes the element
    scale = drop_scale(0.3)
    P = _alloc_planes(ops, rows, cols, "fp32")
    f32 = torch.full((max(rows, 1), cols), float("nan"), device=DEV)[:rows]
    part = ops.split_planes(x, P, relu_mask=mask, colsum=True, mask_scale=scale, out_f32=f32)
    v = torch.where(mask > 0, x, 0.0) * np.float32(scale)
    hi, lo = _split_ref(v)
    assert torch.equal(P[0], hi) and torch.equal(P[1], lo)
    assert torch.equal(f32, v)
    gb = ops.reduce_partials(part)
    ref = v.double().sum(0)
    _check("split_planes colsum", gb, ref, (rows + 4) * U * v.double().abs().sum(0), f"rows={rows} cols={cols}")
    if rows:                                             # without a mask: no scale
        Q = ops.alloc_planes(rows, cols, "bf16", DEV)
        ops.split_planes(x, Q, mask_scale=scale)
        assert torch.equal(Q[0], x.to(torch.bfloat16))


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("K1,K2,N", [(60, 8, 20), (100, 0, 132), (256, 4, 1024)])
def test_weight_planes_bitwise(ops, mode, K1, K2, N):
    g = _gen(K1 + N)
    W1, W2 = _random((K1, N), g), (_random((K2, N), g) if K2 else None)
    W = torch.cat([W1, W2]) if K2 else W1
    hi, lo = _split_ref(W)
    ctr = torch.tensor([(3 << 32) + 5], dtype=torch.int64, device=DEV)
    wp = ops.prepare_weights(W1, W2, mode, dropout_ctr=ctr)
    assert int(ctr) == (3 << 32) + 6                     # one step per call
    ph, pl = _wplanes(wp, K1 + K2, N, mode)
    assert torch.equal(ph[:, :N], hi) and bool((ph[:, N:] == 0).all())
    if mode == "fp32":
        assert torch.equal(pl[:, :N], lo) and bool((pl[:, N:] == 0).all())
    # the per-call forward converts W^T into [n_pad, k_pad] planes of the workspace (zero padded), and advances the
    # dropout counter once
    A = _planes(ops, [_random((5, K1 + K2), g)], mode)
    ops.transform_fwd(A, K1 + K2, 0, W, None, None, True, mode, 0.5, 1, ctr)
    assert int(ctr) == (3 << 32) + 7
    nt, bn = tile_n(N, 32, KBN)
    n_pad, k_pad = nt * bn, _ru(K1 + K2, BK)
    ws = ops._workspace(torch.device(DEV), 0)
    off = _ru(ws.data_ptr(), 1024) - ws.data_ptr()
    plane = n_pad * k_pad * 2
    th = ws[off:off + plane].view(torch.bfloat16).view(n_pad, k_pad)
    want = torch.zeros(n_pad, k_pad, dtype=torch.bfloat16, device=DEV)
    want[:N, :K1 + K2] = hi.t()
    assert torch.equal(th, want)
    if mode == "fp32":
        tl = ws[off + plane:off + 2 * plane].view(torch.bfloat16).view(n_pad, k_pad)
        want[:N, :K1 + K2] = lo.t()
        assert torch.equal(tl, want)


# =========================================================================================================================
# b. forward through both entry points
# =========================================================================================================================
FWD = [  # (M, K1, K2, d_out)
    (1, 4, 0, 4),
    (127, 40, 20, 20),           # K = 60
    (128, 32, 32, 96),           # K = 64
    (129, 36, 32, 132),          # K = 68; BN 96 x 2
    (4097, 1000, 28, 200),       # K = 1,028; BN 224 on the wide tiles
    (130, 512, 512, 256),        # K = 1,024
    (300, 60, 8, 260),           # BN 96 x 3; BN 160 on the wide tiles
    (257, 64, 4, 512),
    (129, 20, 40, 1024),         # global-memory bias, 4 / 8 tiles
    (129, 44, 20, 64),           # BN 64
    (40000, 48, 16, 96),         # more tiles than SMs: both TMEM accumulators alternate within a CTA
    (20000, 56, 8, 256),         # 256 / 128 wide tiles without the narrow-small rule
    (9729, 60, 4, 128),
]


def _fwd_ref(ops, A, P, W, Wp, b, relu, mode, keep=None, scale=None):
    acc, S, T = _prod(P[0], P[1], Wp[0], Wp[1], mode)
    return _epilogue_ref(acc, S, T, b, relu, scale, keep)


def _weights(kind, K1, K2, N, g):
    W1 = _vals(kind, (K1, N), g)
    W2 = _vals(kind, (K2, N), g) if K2 else None
    if kind == "random":
        W1 = W1 / (K1 + K2) ** 0.5
        W2 = None if W2 is None else W2 / (K1 + K2) ** 0.5
    return W1, W2, (torch.cat([W1, W2]) if K2 else W1)


@pytest.mark.parametrize("case", FWD, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("entry", ["fwd", "fwd_w"])
def test_forward(ops, entry, mode, case):
    M, K1, K2, N = case
    g = _gen(M + K1 + N)
    for kind in ("exact", "random"):
        A1 = _vals(kind, (M, K1), g)
        A2 = _vals(kind, (M, K2), g) if K2 else None
        P = _planes(ops, [A1] + ([A2] if K2 else []), mode)
        W1, W2, W = _weights(kind, K1, K2, N, g)
        Wp = _split_ref(W)
        b = _bias(kind, N, g)
        wp = ops.prepare_weights(W1, W2, mode) if entry == "fwd_w" else None
        for relu, bias in ((False, None), (True, b)):
            if entry == "fwd":
                out = ops.transform_fwd(P, K1, K2, W1, W2, bias, relu, mode)
            else:
                out = ops.transform_fwd_w(P, K1 + K2, wp, N, bias, relu, mode)
            ref, bound = _fwd_ref(ops, None, P, W, Wp, bias, relu, mode)
            what = f"{entry} {mode} {case} relu={relu} bias={bias is not None}"
            if kind == "exact":
                _check_exact("forward exact", out, ref, what)
            else:
                _check(f"forward {mode}", out, ref, bound, what)


# =========================================================================================================================
# c. dgrad through both entry points
# =========================================================================================================================
DGRAD = [  # (M, K1, K2, d_out): gA [M, K1 + K2] = G [M, d_out] @ W^T
    (129, 32, 16, 20),           # N = 48
    (4097, 96, 16, 132),         # N = 112
    (300, 256, 4, 64),           # N = 260
    (1000, 768, 256, 256),       # N = 1,024
    (1, 48, 0, 4),
    (40000, 96, 16, 64),
]


@pytest.mark.parametrize("case", DGRAD, ids=lambda c: "x".join(map(str, c)))
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("entry", ["dgrad", "dgrad_w"])
def test_dgrad(ops, entry, mode, case):
    M, K1, K2, N = case
    g = _gen(M + K1 + N + 1)
    for kind in ("exact", "random"):
        G = _planes(ops, [_vals(kind, (M, N), g)], mode)
        W1, W2, W = _weights(kind, K1, K2, N, g)
        Wh, Wl = _split_ref(W)
        wp = ops.prepare_weights(W1, W2, mode) if entry == "dgrad_w" else None
        gA = ops.transform_dgrad(G, N, W1, W2, mode, w_planes=wp)
        acc, S, T = _prod(G[0], G[1], Wh.t(), None if Wl is None else Wl.t(), mode)
        what = f"{entry} {mode} {case}"
        if kind == "exact":
            _check_exact("dgrad exact", gA, acc, what)
        else:
            _check(f"dgrad {mode}", gA, acc, (T + 3) * E23 * S, what)


# =========================================================================================================================
# d. wgrad and g_bias
# =========================================================================================================================
def _wgrad_cases(sm):
    """(rows, K1, K2, d_out, why) from the split rule: 1 split, the 64-split cap, a partial and an empty last split,
    fewer rows than WG_BK, none, and a 128-row m-tile that straddles the W1 / W2 boundary."""
    cases = [(100, 48, 16, 64, "one split"), (20, 36, 12, 20, "rows < WG_BK"), (0, 32, 0, 32, "no rows"),
             (1000, 100, 60, 132, "m-tile straddles W1 / W2"), (3001, 96, 16, 64, "partial last split"),
             (8224, 64, 32, 64, "64-split cap, empty last splits"), (700, 200, 60, 260, "two ragged n tiles")]
    out = []
    for rows, K1, K2, N, why in cases:
        nt, bn = tile_n(N, 64)
        tiles = (K1 + K2 + BM - 1) // BM * nt
        s = wgrad_splits(rows, tiles, sm)
        nps = max(_ru((rows + s - 1) // s, WG_BK), WG_BK)
        out.append((rows, K1, K2, N, why, s, nps))
    return out


@pytest.mark.parametrize("mode", MODES)
def test_wgrad(ops, mode):
    sm = _sm()
    cases = _wgrad_cases(sm)
    reasons = {c[4]: c for c in cases}
    # the cases reach what they claim
    assert reasons["one split"][5] == 1 and reasons["64-split cap, empty last splits"][5] == 64
    r, *_, s, nps = reasons["64-split cap, empty last splits"]
    assert (s - 1) * nps >= r
    r, *_, s, nps = reasons["partial last split"]
    assert s > 1 and 0 < r - (s - 1) * nps < nps and (r - (s - 1) * nps) % WG_BK
    for rows, K1, K2, N, why, s, nps in cases:
        g = _gen(rows + K1 + N)
        for kind in ("exact", "random"):
            A1 = _vals(kind, (rows, K1), g)
            A2 = _vals(kind, (rows, K2), g) if K2 else None
            Gm = _vals(kind, (rows, N), g)
            if kind == "exact" and rows > 1000:
                # sparse rows keep every output below ~1,000 terms (exact accumulation)
                A1 = A1 * (torch.rand(rows, 1, generator=g, device=DEV) < 1000 / rows / 1.5)
            A = _planes(ops, [A1] + ([A2] if K2 else []), mode)
            G = _alloc_planes(ops, rows, N, mode)
            part = ops.split_planes(Gm, G, colsum=True)
            gW1, gW2, gb = ops.transform_wgrad(A, K1, K2, G, N, part, mode)
            acc, S, T = _prod(A[0].t(), None if A[1] is None else A[1].t(), G[0], G[1], mode)
            got = torch.cat([gW1, gW2]) if K2 else gW1
            what = f"{mode} rows={rows} K={K1}+{K2} N={N} ({why}, {s} splits of {nps})"
            gb_ref = Gm.double().sum(0)
            if kind == "exact":
                _check_exact("wgrad exact", got, acc, what)
                _check_exact("wgrad g_bias exact", gb, gb_ref, what)
            else:
                _check(f"wgrad {mode}", got, acc, (T + 3) * E23 * S, what)
                _check("wgrad g_bias", gb, gb_ref, (rows + 4) * U * Gm.double().abs().sum(0), what)
            again = ops.transform_wgrad(A, K1, K2, G, N, part, mode)
            assert torch.equal(gW1, again[0]) and torch.equal(gb, again[2]), what
            if K2:
                assert torch.equal(gW2, again[1]), what


# =========================================================================================================================
# e. fused dropout, element for element;  f. output placement
# =========================================================================================================================
# d_out values that reach every BN class of the store loops (with M = 9,729 the narrow-small rule stays off)
DROP_N = [20, 64, 96, 132, 128, 200, 192, 256, 260]


@pytest.mark.parametrize("p", [0.5, 0.1, 1e-6, 0.99999])
@pytest.mark.parametrize("mode", MODES)
def test_fused_dropout_mask(ops, mode, p):
    """relu(A @ W + b) with the fused dropout, exact operands: bitwise equal to the reference with the ported hash, for
    the per-call and the prepared-weight forward; the counter the GEMM read is the one after the conversion's step."""
    seed = 0x9E3779B9 + int(p * 1000)
    scale = drop_scale(p)
    for N in DROP_N if p == 0.5 else DROP_N[::3]:
        M, K = 9729, 64
        g = _gen(N)
        P = _planes(ops, [_exact((M, K), g)], mode)
        W = _exact((K, N), g)
        b = _bias("exact", N, g)
        for entry in ("fwd", "fwd_w"):
            ctr = torch.tensor([(1 << 32) * 7 + 11], dtype=torch.int64, device=DEV)
            if entry == "fwd":
                out = ops.transform_fwd(P, K, 0, W, None, b, True, mode, p, seed, ctr)
            else:
                wp = ops.prepare_weights(W, None, mode, dropout_ctr=ctr)
                out = ops.transform_fwd_w(P, K, wp, N, b, True, mode, p, seed, ctr)
            c = int(ctr)
            assert c == (1 << 32) * 7 + 12
            keep = drop_keep(M, 0, N, p, seed, c)
            ref, _ = _fwd_ref(ops, None, P, W, _split_ref(W), b, True, mode, keep, scale)
            # the kept values are exact before the scale: one fp32 rounding of the product
            _check_exact("dropout exact", out, ref.float().double(), f"{entry} {mode} p={p} N={N}")
            if p == 0.5:
                frac = float(keep.float().mean())
                assert 0.49 < frac < 0.51


@pytest.mark.parametrize("row_offset", [0, (1 << 24) - 100, (1 << 24) + 3])
@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("mode", MODES)
def test_output_placement(ops, mode, p, row_offset):
    """A column slice of a NaN-filled buffer (ldo > N) and a row window written via ``out=`` and ``row_offset``: the
    written region equals the reference, everything else stays NaN.  Offsets of 2^24 - 100 and 2^24 + 3 rows at N = 256
    put the element indices across and beyond 2^32 (the dropout's block-key branch)."""
    M, K, N = 300, 68, 256
    g = _gen(row_offset % 1000 + 3)
    P = _planes(ops, [_exact((M, K), g)], mode)
    W = _exact((K, N), g)
    b = _bias("exact", N, g)
    seed = 1234
    ctr = torch.tensor([41], dtype=torch.int64, device=DEV)
    wp = ops.prepare_weights(W, None, mode, dropout_ctr=ctr)
    keep = drop_keep(M, row_offset, N, p, seed, int(ctr)) if p else None
    ref, _ = _fwd_ref(ops, None, P, W, _split_ref(W), b, True, mode, keep, 2.0 if p else None)
    # column slice: ldo = N + 12
    buf = torch.full((M + 2, N + 12), float("nan"), device=DEV)
    ops.transform_fwd_w(P, K, wp, N, b, True, mode, p, seed, ctr, row_offset=row_offset, out=buf[1:M + 1, 4:4 + N])
    _check_exact("placement exact", buf[1:M + 1, 4:4 + N], ref, f"column slice {mode} p={p} off={row_offset}")
    rest = buf.clone()
    rest[1:M + 1, 4:4 + N] = float("nan")
    assert bool(rest.isnan().all()), "the forward wrote outside its column slice"
    # row window [100, 100 + 150) of a larger buffer
    big = torch.full((M + 50, N), float("nan"), device=DEV)
    r0, r1 = 100, 250
    ops.transform_fwd_w((P[0][r0:r1], None if P[1] is None else P[1][r0:r1]), K, wp, N, b, True, mode, p, seed, ctr,
                        row_offset=row_offset + r0, out=big[r0:r1])
    _check_exact("placement exact", big[r0:r1], ref[r0:r1], f"row window {mode} p={p} off={row_offset}")
    assert bool(big[:r0].isnan().all()) and bool(big[r1:].isnan().all()), "the forward wrote outside its row window"


# =========================================================================================================================
# g. the run-time store loop (XF = 2): bf16 copy and scattered rows
# =========================================================================================================================
@pytest.mark.parametrize("mode", MODES)
def test_bf16_copy(ops, mode):
    for N in DROP_N:
        M, K = 9729, 60
        g = _gen(N + 5)
        for kind in ("exact", "random"):
            P = _planes(ops, [_vals(kind, (M, K), g)], mode)
            W1, _, W = _weights(kind, K, 0, N, g)
            b = _bias(kind, N, g)
            wp = ops.prepare_weights(W1, None, mode)
            o16 = ops.alloc_planes(M, N, "bf16", DEV)[0]
            out = ops.transform_fwd_w(P, K, wp, N, b, True, mode, out_bf16=o16)
            assert torch.equal(o16, out.to(torch.bfloat16)), (mode, N, kind)
            ref, bound = _fwd_ref(ops, None, P, W, _split_ref(W), b, True, mode)
            if kind == "exact":
                _check_exact("bf16 copy exact", out, ref, f"{mode} N={N}")
            else:
                _check(f"bf16 copy {mode}", out, ref, bound, f"{mode} N={N}")


@pytest.mark.parametrize("use_slot", [False, True])
@pytest.mark.parametrize("mode", MODES)
def test_scattered_rows(ops, lib, mode, use_slot):
    """``rgcn_transform_fwd_w_rows``: row c of the product goes to out[rows[c]] for c < n_list; with ``slot`` only the
    first position of a duplicated node is stored; unlisted rows and the padding rows stay untouched (NaN)."""
    from primekg_rgcn_linkprediction_b200.graph import _ptr, _stream
    n_nodes, K = 5000, 64
    g = _gen(17)
    for N in (20, 132, 256):
        rows = torch.randint(0, n_nodes, (300,), generator=g, device=DEV)
        rows[10:20] = rows[0:10]                         # duplicates
        n_list, n_rows = rows.numel(), rows.numel() + 37  # 37 padding rows of the operand
        Am = _exact((n_rows, K), g)
        first = {}
        for c, r in enumerate(rows.tolist()):
            first.setdefault(r, c)
        first_pos = torch.tensor([first[r] for r in rows.tolist()], device=DEV)
        if not use_slot:
            Am[:n_list] = Am[first_pos]                  # duplicates write identical values
        P = _planes(ops, [Am], mode)
        W = _exact((K, N), g)
        b = _bias("exact", N, g)
        wp = ops.prepare_weights(W, None, mode)
        slot = torch.full((n_nodes,), n_list, dtype=torch.int32, device=DEV)
        slot[rows[first_pos.unique()]] = first_pos.unique().to(torch.int32)
        out = torch.full((n_nodes, N), float("nan"), device=DEV)
        rc = lib.rgcn_transform_fwd_w_rows(_ptr(P[0]), _ptr(P[1]), P[0].stride(0), K, _ptr(wp), _ptr(b), 1, n_rows, N,
                                           _ptr(out), out.stride(0), 0 if mode == "fp32" else 1, _ptr(rows), n_list,
                                           _ptr(slot) if use_slot else None, None, 0, 0, 0, _stream(torch.device(DEV)))
        assert rc == 0
        ref, _ = _fwd_ref(ops, None, P, W, _split_ref(W), b, True, mode)
        listed = torch.zeros(n_nodes, dtype=torch.bool, device=DEV)
        listed[rows] = True
        _check_exact("scattered rows exact", out[rows], ref[first_pos], f"{mode} N={N} slot={use_slot}")
        assert bool(out[~listed].isnan().all())


# =========================================================================================================================
# h. variants selected by environment variables, one child process each
# =========================================================================================================================
VARIANT_CASES = [  # (entry, mode, M, K, N, p, kind)
    ("fwd", "fp32", 4097, 68, 132, 0.0, "random"), ("fwd", "bf16", 129, 1024, 260, 0.5, "exact"),
    ("fwd_w", "fp32", 4097, 68, 260, 0.0, "random"), ("fwd_w", "bf16", 300, 64, 200, 0.5, "exact"),
    ("fwd_w", "fp32", 1000, 1024, 256, 0.0, "random"), ("fwd_w", "bf16", 1000, 1024, 256, 0.0, "random"),
    ("fwd_w", "fp32", 129, 60, 512, 0.5, "exact"), ("fwd_w", "bf16", 4097, 64, 128, 0.0, "exact"),
    ("dgrad_w", "fp32", 2000, 260, 0, 0.0, "random"), ("dgrad_w", "bf16", 300, 1024, 0, 0.0, "exact"),
]


def _variant_outputs():
    """Outputs of VARIANT_CASES, deterministic for a given library and environment."""
    import __graft_entry__ as entry_mod
    entry_mod.build()
    from primekg_rgcn_linkprediction_b200 import ops
    outs = []
    for i, (entry, mode, M, K, N, p, kind) in enumerate(VARIANT_CASES):
        g = _gen(100 + i)
        if entry == "dgrad_w":
            d = 132
            G = _planes(ops, [_vals(kind, (M, d), g)], mode)
            W = _vals(kind, (K, d), g)
            outs.append(ops.transform_dgrad(G, d, W, None, mode, w_planes=ops.prepare_weights(W, None, mode)).cpu())
            continue
        P = _planes(ops, [_vals(kind, (M, K), g)], mode)
        W = _vals(kind, (K, N), g)
        b = _bias(kind, N, g)
        ctr = torch.tensor([5], dtype=torch.int64, device=DEV)
        if entry == "fwd":
            outs.append(ops.transform_fwd(P, K, 0, W, None, b, True, mode, p, 77, ctr).cpu())
        else:
            wp = ops.prepare_weights(W, None, mode, dropout_ctr=ctr)
            outs.append(ops.transform_fwd_w(P, K, wp, N, b, True, mode, p, 77, ctr).cpu())
    return outs


def _variant_refs(outs_len):
    from primekg_rgcn_linkprediction_b200 import ops
    refs = []
    for i, (entry, mode, M, K, N, p, kind) in enumerate(VARIANT_CASES[:outs_len]):
        g = _gen(100 + i)
        if entry == "dgrad_w":
            d = 132
            Gm = _vals(kind, (M, d), g)
            G = _planes(ops, [Gm], mode)
            W = _vals(kind, (K, d), g)
            Wh, Wl = _split_ref(W)
            acc, S, T = _prod(G[0], G[1], Wh.t(), None if Wl is None else Wl.t(), mode)
            refs.append((acc, (T + 3) * E23 * S))
            continue
        P = _planes(ops, [_vals(kind, (M, K), g)], mode)
        W = _vals(kind, (K, N), g)
        b = _bias(kind, N, g)
        keep = drop_keep(M, 0, N, p, 77, 6) if p else None
        refs.append(_fwd_ref(ops, None, P, W, _split_ref(W), b, True, mode, keep, drop_scale(p) if p else None))
    return refs


def _run_variant(env_var, value):
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "out.pt")
        env = dict(os.environ)
        env[env_var] = value
        r = subprocess.run([sys.executable, os.path.abspath(__file__), path], cwd=ROOT, env=env, capture_output=True,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stdout + r.stderr
        return torch.load(path)


@pytest.mark.parametrize("env_var,value,same_bits", [
    ("RGCN_TMA_STORE", "0", True), ("RGCN_GENERIC_EPILOGUE", "1", True),
    ("RGCN_WIDE_TILES", "0", False), ("RGCN_WIDE_FP32", "1", False), ("RGCN_NARROW_SMALL", "0", False)])
def test_environment_variants(ops, env_var, value, same_bits):
    """Store-loop variants must reproduce the default process's bits (same accumulator, same epilogue arithmetic); the
    tile-width variants must give exact cases bitwise and random cases within the bound."""
    default = _variant_outputs()
    got = _run_variant(env_var, value)
    refs = _variant_refs(len(default))
    bitwise = []
    for case, d, o, (ref, bound) in zip(VARIANT_CASES, default, got, refs):
        what = f"{env_var}={value} {case}"
        if same_bits:
            assert torch.equal(d, o), what
        elif case[-1] == "exact":
            _check_exact("variants exact", o.to(DEV), ref, what)
        else:
            _check(f"variants {case[1]}", o.to(DEV), ref, bound, what)
            bitwise.append(bool(torch.equal(d, o)))
    if bitwise:
        print(f"\n[gemm conformance] {env_var}={value}: random cases bitwise equal to the default: {bitwise}", end="")


# =========================================================================================================================
# i. consuming epilogues: threshold (diagonal tiles) and rank counts
# =========================================================================================================================
@pytest.mark.parametrize("d", [4, 20, 256])
@pytest.mark.parametrize("nq", [1, 127, 129])
def test_scores_rank_counts(ops, lib, nq, d):
    """``rgcn_scores_diag_w`` thresholds bitwise equal to the materialised tensor-core score matrix of the same planes,
    and ``rgcn_scores_rank_w`` counts equal to the counts taken from that matrix; duplicated candidates give exact ties
    and one true tail sits at the last column."""
    from primekg_rgcn_linkprediction_b200.graph import _ptr, _stream
    from primekg_rgcn_linkprediction_b200.rank import scores_from_rows
    g = _gen(nq * 31 + d)
    for nc in (1, 129, 1025, 5593, 30926):
        A = torch.randn(nq, d, generator=g, device=DEV)
        C = torch.randn(nc, d, generator=g, device=DEV)
        if nc > 2:
            C[nc // 2] = C[nc // 3]                      # an exact duplicate candidate
        tails = torch.randint(0, nc, (nq,), generator=g, device=DEV)
        tails[0] = nc - 1
        if nc > 2 and nq > 1:
            tails[1] = nc // 3                           # a true tail with an exact tie
        Q = ops.alloc_planes(nq, d, "fp32", DEV)
        ops.split_planes(A, Q)
        cand_planes = ops.prepare_weights(C, None, "fp32")
        tail_planes = ops.prepare_weights(C[tails].contiguous(), None, "fp32")
        thr = torch.empty(nq, dtype=torch.float32, device=DEV)
        greater = torch.zeros(nq, dtype=torch.int32, device=DEV)
        equal = torch.zeros(nq, dtype=torch.int32, device=DEV)
        st = _stream(torch.device(DEV))
        assert lib.rgcn_scores_diag_w(_ptr(Q[0]), _ptr(Q[1]), Q[0].stride(0), d, _ptr(tail_planes), nq, _ptr(thr), st) == 0
        assert lib.rgcn_scores_rank_w(_ptr(Q[0]), _ptr(Q[1]), Q[0].stride(0), d, _ptr(cand_planes), nc, nq, _ptr(thr),
                                      _ptr(tails), _ptr(greater), _ptr(equal), st) == 0
        S = scores_from_rows(A, C, method="tc")
        st_ = S.gather(1, tails.view(-1, 1))
        assert torch.equal(thr, st_.view(-1)), (nq, nc, d)
        others = torch.ones_like(S, dtype=torch.bool)
        others.scatter_(1, tails.view(-1, 1), False)
        assert torch.equal(greater.long(), ((S > st_) & others).sum(1)), (nq, nc, d)
        assert torch.equal(equal.long(), ((S == st_) & others).sum(1)), (nq, nc, d)
        if nc > 2 and nq > 1:
            assert int(equal[1]) >= 1


# =========================================================================================================================
# coverage of the kernel instantiations
# =========================================================================================================================
def test_cases_reach_every_instantiation():
    """Every (SPLIT, B_MN, BNT, XF, BN class) the default launch code can select is reached by the cases above."""
    sm = _sm()
    reachable = set()
    for split in (True, False):
        for bn in range(32, 257, 32):
            cls, bnt = bn_class(bn), (256 if bn > 128 else 128)
            if bn <= 128:
                reachable |= {(split, False, 128, xf, cls) for xf in (0, 1)}   # per-call forward (dgrad: xf 0)
            reachable.add((split, False, bnt, 0, cls))                        # dgrad_w: wide tiles for K > 128
            if bn <= 128 or not split:                                        # fp32 mode: 128-wide tiles only
                reachable |= {(split, True, bnt, xf, cls) for xf in (0, 1, 2)}  # prepared-weight forward
    reached = set()

    def add(entry, mode, M, K, N, xf):
        s, b_mn, bnt, x, bn = launch_choice(entry, mode, M, K, N, xf, sm)
        reached.add((s, b_mn, bnt, x, bn_class(bn)))

    for mode in MODES:
        for M, K1, K2, N in FWD:
            add("fwd", mode, M, K1 + K2, N, 0)
            add("fwd_w", mode, M, K1 + K2, N, 0)
        for M, K1, K2, N in DGRAD:
            add("dgrad", mode, M, K1 + K2, N, 0)
            add("dgrad_w", mode, M, K1 + K2, N, 0)
        for N in DROP_N:
            add("fwd", mode, 9729, 64, N, 1)
            add("fwd_w", mode, 9729, 64, N, 1)
            add("fwd_w", mode, 9729, 60, N, 2)
    missing = reachable - reached
    assert not missing, sorted(missing)
    assert reached <= reachable, sorted(reached - reachable)


if __name__ == "__main__":
    # child process of test_environment_variants: python test_gpu_gemm_conformance.py OUT.pt
    sys.path.insert(0, ROOT)
    torch.save(_variant_outputs(), sys.argv[1])
