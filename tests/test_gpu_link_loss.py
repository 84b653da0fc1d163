"""The fused decoder + loss (csrc/decoder.cu: link_loss_fwd_kernel, link_contrib_kernel, link_gather_kernel and the
relation-table partial reduction) against a float64 reference built from plain torch ops on the device.

The reference covers the DistMult score with the relation dropout, the BCE-with-logits loss, the accuracy count of the
reference training script (``sigmoid(s) > 0.5`` on the kernel's own fp32 score) and the gradients with respect to the
node embeddings and the relation table.  The dropout multipliers come from a port of the counter hash of decoder.cu
(``pcg32`` / ``rel_drop4``): that hash, not torch's Philox stream, is the project's definition of the mask.

Tolerances follow from the operation, not from a flat ``atol * max``: an output that is a sum of K terms must satisfy
``|got - ref| <= (K + 4) * 2^-24 * sum |terms|`` with the terms in float64, so an unlisted gradient row, an unused
relation or a fully dropped element must be exactly zero.  Where the per-pair gradient is itself computed by the
kernel (``link_loss``'s backward), its own rounding error is added to the bound.  The hub cases use small integers and
must match the reference exactly: at K >= 1,000 the worst-case bound no longer resolves one missing term.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -24                       # unit roundoff of fp32
ETA = 2.0 ** -149                    # smallest fp32 subnormal: the absolute rounding error below the normal range
M32 = 0xFFFFFFFF

# Branch thresholds of csrc/decoder.cu (rgcn_link_loss_bwd_rows and link_gather_kernel):
SMEM_LIST_BYTES = 200 * 1024         # the 2 n positions (in windows of 128 ints) are scanned from shared memory up to this
LIST_WINDOW = 128                    # shared-memory scan window, in positions
LINK_LIST = 128                      # kLinkList: positions an owner collects before it adds them
PASS_FLOATS = 256                    # a gather column pass covers 64 float4 per row
DEFAULT_SMEM = 48 * 1024             # CUDA's per-block limit (static + dynamic) without an opt-in
GATHER_STATIC_SMEM = 8 * LINK_LIST * 4 + 32 * 4   # s_list + s_r of link_gather_kernel


def _list_bytes(n):
    return (2 * n + LIST_WINDOW - 1) // LIST_WINDOW * LIST_WINDOW * 4


def _scan_in_smem(n):
    return _list_bytes(n) <= SMEM_LIST_BYTES


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


# ---- float64 reference ------------------------------------------------------------------------------------------------
def _pcg32(x):
    state = (x * 747796405 + 2891336453) & M32
    word = (((state >> ((state >> 28) + 4)) ^ state) * 277803737) & M32
    return ((word >> 22) ^ word) & M32


def _drop_mult(n, d, p, seed, c):
    """[n, d] float64 multipliers (0 or float32(1 / (1 - p))) of the relation dropout of the call that read counter c."""
    if p == 0.0:
        return None
    pf = np.float32(p)                                   # the C ABI takes p as a float
    thresh = max(1, int(float(pf) * 65536.0 + 0.5))
    scale = float(np.float32(1.0) / (np.float32(1.0) - pf))
    key = (_pcg32((seed & M32) ^ (c & M32)) + ((c >> 32) * 0x9E3779B9)) & M32
    pi = torch.arange(n, device=DEV, dtype=torch.int64)[:, None]
    e = (pi * d + 4 * torch.arange(d // 4, device=DEV, dtype=torch.int64)[None, :]) & M32
    h0, h1 = _pcg32(e ^ key), _pcg32(((e + 2) & M32) ^ key)
    bits = torch.stack([h0 & 0xFFFF, h0 >> 16, h1 & 0xFFFF, h1 >> 16], dim=2).reshape(n, d)
    return torch.where(bits >= thresh, scale, 0.0).to(torch.float64)


class Ref:
    """Scores and gradients of one call in float64; invalid pairs (an index out of range) contribute nothing."""

    def __init__(self, emb, table, head, tail, rel, mult):
        N, R = emb.size(0), table.size(0)
        self.N, self.R = N, R
        self.valid = (head >= 0) & (head < N) & (tail >= 0) & (tail < N) & (rel >= 0) & (rel < R)
        z = torch.zeros_like(head)
        self.hs, self.ts, self.rs = (torch.where(self.valid, x, z) for x in (head, tail, rel))
        E, W = emb.detach().double(), table.detach().double()
        self.mult = mult
        self.H, self.T = E[self.hs], E[self.ts]
        self.Rm = W[self.rs] if mult is None else W[self.rs] * mult
        terms = self.H * self.Rm * self.T
        d = emb.size(1)
        self.s = terms.sum(1)
        self.s_bound = (d + 4) * U * terms.abs().sum(1) + 4 * d * ETA

    def grads(self, g, gerr=None):
        """(g_emb, bound, g_tab, bound) for per-pair gradients g (float64 [n]); gerr: error bound of a kernel-computed g."""
        v = self.valid
        g = torch.where(v, g, 0.0)
        m = torch.ones_like(self.Rm) if self.mult is None else self.mult
        ch, ct = g[:, None] * self.Rm * self.T, g[:, None] * self.H * self.Rm
        cr = g[:, None] * self.H * self.T * m
        d = self.H.size(1)
        hs, ts, rs = self.hs[v], self.ts[v], self.rs[v]

        def scatter(rows, n_rows, *vals):
            out = torch.zeros(n_rows, d, dtype=torch.float64, device=DEV)
            for r, x in zip(rows, vals):
                out.index_add_(0, r, x[v])
            return out

        k_emb = torch.bincount(torch.cat([hs, ts]), minlength=self.N).double()[:, None]
        k_tab = torch.bincount(rs, minlength=self.R).double()[:, None]
        g_emb = scatter((hs, ts), self.N, ch, ct)
        b_emb = (k_emb + 4) * U * scatter((hs, ts), self.N, ch.abs(), ct.abs()) + 4 * k_emb * ETA
        g_tab = scatter((rs,), self.R, cr)
        b_tab = (k_tab + 4) * U * scatter((rs,), self.R, cr.abs()) + 4 * k_tab * ETA
        if gerr is not None:
            e = torch.where(v, gerr, 0.0)[:, None]
            b_emb += scatter((hs, ts), self.N, e * (self.Rm * self.T).abs(), e * (self.H * self.Rm).abs())
            b_tab += scatter((rs,), self.R, e * (self.H * self.T * m).abs())
        return g_emb, b_emb, g_tab, b_tab


def _ratio(got, ref, bound, what):
    """Worst |got - ref| / bound; an error where the bound is 0, or a NaN, counts as infinite."""
    err = (got.detach().double() - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / bound)
    r = float(torch.nan_to_num(r, nan=float("inf")).max()) if r.numel() else 0.0
    assert r <= 1.0, f"{what}: error / bound = {r:.3g} (worst element at {int((err / bound).nan_to_num(float('inf')).argmax())})"
    return r


def _exact(got, ref, what):
    got = got.detach().double()
    assert torch.equal(got, ref), f"{what}: {int((got != ref).sum())} elements differ from the exact reference"
    return 0.0


# ---- inputs -----------------------------------------------------------------------------------------------------------
def _sampled(n, N, R, gen):
    """Positives with a skewed node distribution (low ids are hubs) and three corruptions each that keep one end, as
    the negative sampler makes them; relation R - 1 is never used."""
    npos = (n + 3) // 4
    ph = (N * torch.rand(npos, generator=gen) ** 3).long().clamp_max(N - 1)
    pt = (N * torch.rand(npos, generator=gen) ** 3).long().clamp_max(N - 1)
    pr = torch.randint(0, R - 1, (npos,), generator=gen)
    keep_h = torch.rand(npos, 3, generator=gen) < 0.5
    ent = torch.randint(0, N, (npos, 3), generator=gen)
    nh = torch.where(keep_h, ph[:, None], ent).reshape(-1)
    nt = torch.where(keep_h, ent, pt[:, None]).reshape(-1)
    h = torch.cat([ph, nh])[:n]
    t = torch.cat([pt, nt])[:n]
    r = torch.cat([pr, pr.repeat_interleave(3)])[:n]
    y = torch.cat([torch.ones(npos), torch.zeros(3 * npos)])[:n]
    return h, t, r, y


def _hubs(n, N, R, gen):
    """Node 0 at exactly LINK_LIST positions, node 1 at LINK_LIST + 1, node 2 at about 1,500 (ten of them self pairs),
    fifty other self pairs h == t; every other position holds a node >= 3."""
    h = torch.randint(3, N, (n,), generator=gen)
    t = torch.randint(3, N, (n,), generator=gen)
    perm = torch.randperm(n, generator=gen)
    hub_self, other_self = perm[:10], perm[10:60]
    t[other_self] = h[other_self]
    h[hub_self] = 2
    t[hub_self] = 2
    taken = torch.zeros(2 * n, dtype=torch.bool)
    taken[perm[:60]] = True
    taken[perm[:60] + n] = True
    free = torch.nonzero(~taken).flatten()
    free = free[torch.randperm(free.numel(), generator=gen)]
    pos = torch.cat([h, t])
    counts = (LINK_LIST, LINK_LIST + 1, 1500 - 20)
    at = 0
    for node, k in enumerate(counts):
        pos[free[at:at + k]] = node
        at += k
    h, t = pos[:n].clone(), pos[n:].clone()
    r = torch.randint(0, R - 1, (n,), generator=gen)
    y = (torch.rand(n, generator=gen) < 0.25).float()
    return h, t, r, y


def _invalid(n, N, R, gen, node0):
    """About 1 % out-of-range heads, tails or relations (parked on row 0 by the backward).  node0 == "hub": node 0 is a
    hub whose first valid position comes after parked ones; "unlisted": no valid pair lists node 0."""
    h, t, r, y = _sampled(n, N, R, gen)
    if node0 == "unlisted":
        h = torch.where(h == 0, 1, h)
        t = torch.where(t == 0, 1, t)
    else:
        h[: n // 2][torch.rand(n // 2, generator=gen) < 0.05] = 0
    bad = torch.nonzero(torch.rand(n, generator=gen) < 0.01).flatten()
    bad = torch.cat([torch.arange(5), bad])                          # the first positions are parked ones
    kind = torch.arange(bad.numel()) % 5
    h[bad[kind == 0]] = N + 7
    t[bad[kind == 1]] = -3
    r[bad[kind == 2]] = R + 2
    r[bad[kind == 3]] = -1
    h[bad[kind == 4]] = -1
    return h, t, r, y


# name: (n, d, N, R, p_drop, inputs, integer)
CASES = {
    "partial_n1_d4": (1, 4, 50, 3, 0.1, "random", False),
    "partial_n7_d4": (7, 4, 50, 3, 0.1, "random", False),
    "partial_n9_d4": (9, 4, 50, 3, 0.1, "random", False),
    "partial_n1_d64": (1, 64, 50, 3, 0.1, "random", False),
    "partial_n7_d64": (7, 64, 50, 3, 0.0, "random", False),
    "partial_n9_d64": (9, 64, 50, 3, 0.1, "random", False),
    "cfg2_shape": (2048, 256, 30926, 3, 0.1, "sampled", False),
    "smem_last_25600": (25600, 64, 30926, 30, 0.1, "sampled", False),
    "global_first_25601": (25601, 64, 30926, 30, 0.1, "sampled", False),
    "global_40960_d256": (40960, 256, 30926, 30, 0.1, "sampled", False),
    "hubs_smem_4096": (4096, 128, 20000, 5, 0.5, "hubs", True),
    "hubs_global_40960": (40960, 128, 20000, 5, 0.5, "hubs", True),
    "one_node_4096": (4096, 128, 100, 5, 0.5, "one_node", True),
    "wide_d260": (512, 260, 3000, 4, 0.5, "sampled", False),
    "wide_d512": (512, 512, 3000, 4, 0.5, "sampled", False),
    "invalid_hub0_2048": (2048, 64, 5000, 5, 0.1, "invalid_hub", False),
    "invalid_unlisted0_2048": (2048, 64, 5000, 5, 0.1, "invalid_unlisted", False),
    "invalid_hub0_30000": (30000, 64, 30926, 5, 0.1, "invalid_hub", False),
    "invalid_unlisted0_30000": (30000, 64, 30926, 5, 0.1, "invalid_unlisted", False),
}


def _inputs(name, seed=0):
    n, d, N, R, p, kind, integer = CASES[name]
    gen = torch.Generator().manual_seed(1000 + seed + sum(map(ord, name)))
    if kind == "random":
        h, t = torch.randint(0, N, (n,), generator=gen), torch.randint(0, N, (n,), generator=gen)
        r, y = torch.randint(0, R - 1, (n,), generator=gen), (torch.rand(n, generator=gen) < 0.5).float()
    elif kind == "sampled":
        h, t, r, y = _sampled(n, N, R, gen)
    elif kind == "hubs":
        h, t, r, y = _hubs(n, N, R, gen)
    elif kind == "one_node":
        h = torch.full((n,), 7)
        t = h.clone()
        r, y = torch.randint(0, R - 1, (n,), generator=gen), (torch.rand(n, generator=gen) < 0.5).float()
    else:
        h, t, r, y = _invalid(n, N, R, gen, "hub" if kind == "invalid_hub" else "unlisted")
    if integer:                                  # every partial sum stays below 2^24: fp32 is exact in any order
        emb = torch.randint(-2, 3, (N, d), generator=gen).float()
        table = torch.randint(-2, 3, (R, d), generator=gen).float()
        coef = torch.randint(-3, 4, (n,), generator=gen).float()
    else:
        emb, table, coef = torch.randn(N, d, generator=gen), torch.randn(R, d, generator=gen), torch.randn(n, generator=gen)
    return dict(emb=emb.to(DEV), table=table.to(DEV), head=h.to(DEV), tail=t.to(DEV), rel=r.to(DEV), y=y.to(DEV),
                coef=coef.to(DEV), p=p, integer=integer, kind=kind)


def _clear_status(ops):
    try:
        ops.raise_on_bad_pairs(torch.device(DEV))
    except IndexError:
        pass


def _check_call(inp, seed=1234, ctr=None, tag=""):
    """One link_loss forward + backward and one pair_scores forward + backward against the reference."""
    from primekg_rgcn_linkprediction_b200 import ops, rowsparse
    emb = inp["emb"].clone().requires_grad_()
    table = inp["table"].clone().requires_grad_()
    h, t, r, y, coef, p = inp["head"], inp["tail"], inp["rel"], inp["y"], inp["coef"], inp["p"]
    n, d = h.numel(), emb.size(1)
    ctr = ops.rng_counter(DEV) if ctr is None else ctr
    out = {}
    exact = inp["integer"]

    # link_loss: scores, loss, accuracy and its backward
    c0 = int(ctr)
    loss, s32, correct = ops.link_loss(emb, table, h, t, r, y, p, seed, ctr)
    assert int(ctr) == c0 + (1 if p > 0 else 0), "the counter advances by one per dropout call"
    ref = Ref(emb, table, h, t, r, _drop_mult(n, d, p, seed, c0))
    v = ref.valid
    assert bool(torch.isnan(s32[~v]).all()), "an invalid pair's score is NaN"
    out["score"] = (_exact(s32[v], ref.s[v], "score") if exact else _ratio(s32[v], ref.s[v], ref.s_bound[v], "score"))
    if bool(v.all()):
        s64 = ref.s
        l64 = s64.clamp_min(0) - s64 * y.double() + torch.log1p(torch.exp(-s64.abs()))
        lb = (n / 256 + 40) * U * float(l64.abs().mean()) + float(ref.s_bound.mean())
        out["loss"] = _ratio(loss.detach().reshape(1), l64.mean().reshape(1), torch.tensor([lb], device=DEV), "loss")
    else:
        assert bool(torch.isnan(loss)), "an invalid pair makes the loss NaN"
    want = int(((torch.sigmoid(s32) > 0.5).float() == y).sum())          # reference src/train.py:321-322
    assert int(correct) == want, f"accuracy count {int(correct)} != {want}"
    g_emb, g_tab = torch.autograd.grad(loss, (emb, table))
    rowsparse.clear()
    sig = torch.sigmoid(s32.double())
    g64 = (sig - y.double()) / n
    # the kernel computes g = (1 / (1 + expf(-s)) - y) / n in fp32: a few roundings relative to sigmoid(s) and |g|, and
    # a sigmoid below the normal range (expf(-s) overflows for s < -88.7) may be lost entirely
    gerr = (8 * U * (sig + (sig - y.double()).abs()) + sig.clamp_max(2.0 ** -126)) / n + ETA
    ge, be, gt, bt = ref.grads(g64, gerr)
    out["loss g_emb"] = _ratio(g_emb, ge, be, "link_loss g_emb")
    out["loss g_tab"] = _ratio(g_tab, gt, bt, "link_loss g_tab")

    # pair_scores driven by fp32 coefficients: the incoming gradient is exact, the bound covers the kernels alone
    c1 = int(ctr)
    s2 = ops.pair_scores(emb, table, h, t, r, p, seed, ctr)
    assert int(ctr) == c1 + (1 if p > 0 else 0)
    ref2 = Ref(emb, table, h, t, r, _drop_mult(n, d, p, seed, c1))
    g_emb2, g_tab2 = torch.autograd.grad((s2 * coef).sum(), (emb, table))
    rowsparse.clear()
    ge, be, gt, bt = ref2.grads(coef.double())
    if exact:
        _exact(s2[v], ref2.s[v], "pair_scores score")
        out["g_emb"] = _exact(g_emb2, ge, "g_emb")
        out["g_tab"] = _exact(g_tab2, gt, "g_tab")
    else:
        out["pair score"] = _ratio(s2[v], ref2.s[v], ref2.s_bound[v], "pair_scores score")
        out["g_emb"] = _ratio(g_emb2, ge, be, "g_emb")
        out["g_tab"] = _ratio(g_tab2, gt, bt, "g_tab")
    listed = torch.zeros(ref.N, dtype=torch.bool, device=DEV)
    listed[ref.hs[v]] = True
    listed[ref.ts[v]] = True
    assert int(torch.count_nonzero(g_emb2[~listed])) == 0, "unlisted gradient rows are exactly zero"
    used = torch.zeros(ref.R, dtype=torch.bool, device=DEV)
    used[ref.rs[v]] = True
    assert not bool(used.all()) and int(torch.count_nonzero(g_tab2[~used])) == 0, "an unused relation's row is exactly zero"
    print(f"{tag} worst error / bound: " + ", ".join(f"{k} {x:.3g}" for k, x in out.items()))
    return dict(s=s32, loss=loss, correct=correct, g_emb=g_emb2, g_tab=g_tab2, valid=v, listed=listed, ref=ref)


@pytest.mark.parametrize("name", list(CASES))
def test_link_loss_against_fp64_reference(pkg, name):
    from primekg_rgcn_linkprediction_b200 import ops
    n, d, N, R, p, kind, integer = CASES[name]
    inp = _inputs(name)
    h, t = inp["head"], inp["tail"]
    pos = torch.cat([h, t])
    # each case reaches the branch it is named for
    if name.startswith("partial"):
        assert n % 8 != 0 and n < 32                                  # partial warps / blocks and 32-pair table chunks
    if name.startswith("smem") or name.endswith("_4096") or name == "cfg2_shape":
        assert _scan_in_smem(n)
    if name.startswith("global") or name.endswith("_40960"):
        assert not _scan_in_smem(n)
    if name.startswith("smem_last"):
        assert not _scan_in_smem(n + 1)
    if kind == "hubs":
        cnt = torch.bincount(pos, minlength=N)
        assert cnt[0] == LINK_LIST and cnt[1] == LINK_LIST + 1 and 1400 < cnt[2] < 1600
        assert bool((h == t).sum() >= 60)
    if kind == "one_node":
        assert bool((pos == pos[0]).all())                            # every scan window is full
    if name.startswith("wide"):
        assert d > PASS_FLOATS                                        # a second column pass
    _clear_status(ops)
    _check_call(inp, tag=name)
    if kind.startswith("invalid"):
        with pytest.raises(IndexError):
            ops.raise_on_bad_pairs(torch.device(DEV))
        if kind == "invalid_hub":
            r = inp["rel"]
            ok = (h >= 0) & (h < N) & (t >= 0) & (t < N) & (r >= 0) & (r < R)
            assert bool(~ok[:5].any()) and int(torch.nonzero(ok & ((h == 0) | (t == 0))).min()) > 4   # parked first
    ops.raise_on_bad_pairs(torch.device(DEV))                        # reported once, or nothing to report


def test_link_loss_accuracy_in_the_sigmoid_band(pkg):
    """With d = 4, h = (x, 0, 0, 0) and r = t = 1 the score is exactly x: logits around 0, where ``s > 0`` and
    ``sigmoid(s) > 0.5`` disagree in fp32, and the extremes, with both labels."""
    from primekg_rgcn_linkprediction_b200 import ops
    x, y = _band_logits()
    m = x.numel()
    emb = torch.zeros(m + 1, 4, device=DEV)
    emb[:m, 0] = x
    emb[m] = 1.0
    table = torch.ones(1, 4, device=DEV)
    idx = torch.arange(m, device=DEV)
    loss, s, correct = ops.link_loss(emb, table, idx, torch.full_like(idx, m), torch.zeros_like(idx), y)
    assert torch.equal(s, x)
    want = int(((torch.sigmoid(s) > 0.5).float() == y).sum())
    assert int(correct) == want, f"accuracy count {int(correct)} != {want}"
    x64 = x.double()
    l64 = x64.clamp_min(0) - x64 * y.double() + torch.log1p(torch.exp(-x64.abs()))
    bound = (m / 256 + 40) * U * float(l64.mean())
    assert abs(float(loss) - float(l64.mean())) <= bound


def _band_logits():
    """A dense sweep of [-2e-7, 2e-7] (labels 1, 0, 0, 1, 0, 0, ...: the two labels do not cancel in the count), then
    +-0, +- the smallest subnormal and +-1e4 with each label."""
    sweep = torch.linspace(-2e-7, 2e-7, 40_001, device=DEV)
    tiny = 2.0 ** -149
    special = torch.tensor([0.0, -0.0, tiny, -tiny, 1e4, -1e4], device=DEV).repeat(2)
    x = torch.cat([sweep, special])
    y = torch.cat([(torch.arange(sweep.numel(), device=DEV) % 3 == 0).float(),
                   torch.tensor([1.0] * 6 + [0.0] * 6, device=DEV)])
    return x, y


def _padded(n_total, gen_seed=5):
    """25,000 real pairs followed by padding pairs of real hub nodes with coefficient 0."""
    n_real, N, R, d = 25_000, 30926, 30, 64
    gen = torch.Generator().manual_seed(gen_seed)
    h, t, r, y = _sampled(n_real, N, R, gen)
    emb, table, coef = torch.randn(N, d, generator=gen), torch.randn(R, d, generator=gen), torch.randn(n_real, generator=gen)
    hubs = torch.bincount(torch.cat([h, t]), minlength=N).argsort(descending=True)[:16]
    gp = torch.Generator().manual_seed(6)
    k = n_total - n_real
    ph, pt = hubs[torch.randint(0, 16, (k,), generator=gp)], hubs[torch.randint(0, 16, (k,), generator=gp)]
    pr = torch.randint(0, R - 1, (k,), generator=gp)
    cat = lambda a, b: torch.cat([a, b]).to(DEV)                      # noqa: E731
    return dict(emb=emb.to(DEV), table=table.to(DEV), head=cat(h, ph), tail=cat(t, pt), rel=cat(r, pr),
                coef=cat(coef, torch.zeros(k)), p=0.1)


def _pair_scores_grads(inp, seed=77):
    from primekg_rgcn_linkprediction_b200 import ops, rowsparse
    emb = inp["emb"].clone().requires_grad_()
    table = inp["table"].clone().requires_grad_()
    ctr = ops.rng_counter(DEV)                                        # every call draws with counter value 0
    s = ops.pair_scores(emb, table, inp["head"], inp["tail"], inp["rel"], inp["p"], seed, ctr)
    g_emb, g_tab = torch.autograd.grad((s * inp["coef"]).sum(), (emb, table))
    rowsparse.clear()
    return s.detach(), g_emb, g_tab


def test_shared_memory_scan_equals_global_scan_bitwise(pkg):
    """Padding at the end keeps the real positions in the same relative order and adds zero contributions, the real
    pairs' table partials fall into the same 32-pair chunks, and the partial reduction only appends zeros: the
    shared-memory scan (n = 25,600) and the global-memory scan (n = 35,000) must give the same bits."""
    assert _scan_in_smem(25_600) and not _scan_in_smem(35_000)
    s_a, ge_a, gt_a = _pair_scores_grads(_padded(25_600))
    s_b, ge_b, gt_b = _pair_scores_grads(_padded(35_000))
    assert torch.equal(s_a[:25_000], s_b[:25_000])
    assert torch.equal(ge_a, ge_b)
    assert torch.equal(gt_a, gt_b)


def test_global_scan_backward_is_bitwise_deterministic(pkg):
    inp = _inputs("global_40960_d256")
    assert not _scan_in_smem(inp["head"].numel())
    a = _pair_scores_grads(inp)
    b = _pair_scores_grads(inp)
    for x, z in zip(a, b):
        assert torch.equal(x, z)


def test_listed_only_backward_equals_full_backward_on_listed_rows(pkg, monkeypatch):
    """``rowsparse.mark_listed_output(emb)`` between the forward and the backward: the backward skips the zero fill of
    the unlisted rows and must leave the listed rows bitwise as the unmarked call does."""
    from primekg_rgcn_linkprediction_b200 import ops, rowsparse
    inp = _inputs("cfg2_shape")
    full = _check_call(inp, tag="listed-only reference")
    seen = []
    real = rowsparse.is_listed_output
    monkeypatch.setattr(rowsparse, "is_listed_output", lambda e: seen.append(real(e)) or seen[-1])
    emb = inp["emb"].clone().requires_grad_()
    table = inp["table"].clone().requires_grad_()
    ctr = ops.rng_counter(DEV)
    ctr.fill_(1)                                                      # the counter value the reference's pair_scores read
    s = ops.pair_scores(emb, table, inp["head"], inp["tail"], inp["rel"], inp["p"], 1234, ctr)
    rowsparse.mark_listed_output(emb)
    g_emb, g_tab = torch.autograd.grad((s * inp["coef"]).sum(), (emb, table))
    rowsparse.clear()
    assert seen == [True], "the backward took the listed-only form"
    lst = full["listed"]
    assert torch.equal(g_emb[lst], full["g_emb"][lst])
    assert torch.equal(g_tab, full["g_tab"])


def _window_case(n):
    """Entry point of the fresh interpreter of the test below."""
    import primekg_rgcn_linkprediction_b200  # noqa: F401
    N, R, d = 30926, 3, 64
    CASES[f"window_{n}"] = (n, d, N, R, 0.1, "sampled", False)
    _check_call(_inputs(f"window_{n}"), tag=f"window n={n}")


@pytest.mark.parametrize("n", [6144, 5569])
def test_gather_shared_memory_opt_in_window(pkg, n):
    """Batches whose position list fits the 48 KB default only without the gather kernel's static shared memory: the
    launch needs the opt-in.  A fresh interpreter, so that no larger batch has raised the limit of the process before."""
    dyn = _list_bytes(n)
    assert dyn <= DEFAULT_SMEM < dyn + GATHER_STATIC_SMEM
    code = (f"import sys; sys.path.insert(0, {ROOT!r}); sys.path.insert(0, {os.path.join(ROOT, 'tests')!r}); "
            f"import test_gpu_link_loss as T; T._window_case({n})")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stdout + r.stderr
