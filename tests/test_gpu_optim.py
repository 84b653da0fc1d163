"""GPU tests of the fused clip + Adam / AdamW step (csrc/optim.cu, optim.FusedAdam) against torch.optim.Adam +
torch.nn.utils.clip_grad_norm_, eagerly and as the last kernels of a captured GraphedTrainStep."""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
# cfg2's parameter shapes with the node table cut to 3,001 rows (an odd count: the table's numel is not a multiple of 4)
SHAPES = [(3001, 64), (3, 64, 256), (64, 256), (256,), (3, 256, 256), (256, 256), (256,), (3, 256), (1003,)]


@pytest.fixture(scope="module")
def pkg(lib_built):
    return lib_built


def _params(seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    ps = [torch.nn.Parameter(torch.randn(s, generator=g, device=DEV) * 0.1) for s in SHAPES]
    # one parameter that is not 16-byte aligned (a view at offset 1): the kernels' scalar path
    base = torch.randn(1 + 999, generator=g, device=DEV) * 0.1
    ps.append(torch.nn.Parameter(base[1:]))
    assert ps[-1].data_ptr() % 16 != 0
    return ps


def _grads(seed, params, scale):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return [torch.randn(p.shape, generator=g, device=DEV) * scale for p in params]


CONFIGS = {  # name: (optimizer kwargs, max_grad_norm, gradient scale)
    "adam_l2_noclip": (dict(weight_decay=1e-2), None, 1e-2),
    "adam_l2_clip_inactive": (dict(weight_decay=1e-2), 1e6, 1e-2),
    "adam_l2_clip_active": (dict(weight_decay=1e-2), 1.0, 1e-1),
    "adamw_noclip": (dict(weight_decay=1e-2, decoupled_weight_decay=True), None, 1e-2),
    "adamw_clip_inactive": (dict(weight_decay=1e-2, decoupled_weight_decay=True), 1e6, 1e-2),
    "adamw_clip_active": (dict(weight_decay=1e-2, decoupled_weight_decay=True), 1.0, 1e-1),
}


def _rel(a, b):
    return float(((a - b).abs() / b.abs().clamp_min(1e-30)).max())


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_fused_adam_matches_torch(pkg, name):
    kw, max_norm, scale = CONFIGS[name]
    ours, ref = _params(1), _params(1)
    opt = pkg.FusedAdam(ours, lr=1e-2, max_grad_norm=max_norm, **kw)
    topt = torch.optim.Adam(ref, lr=1e-2, foreach=False, **kw)
    worst = {"step1": 0.0, "step50": 0.0, "grad_norm": 0.0}
    for it in range(50):
        gs = _grads(100 + it, ours, scale)
        for p, q, g in zip(ours, ref, gs):
            p.grad, q.grad = g.clone(), g.clone()
        if max_norm is not None:
            tn = torch.nn.utils.clip_grad_norm_(ref, max_norm, foreach=False)
        opt.step()
        topt.step()
        if max_norm is not None:
            torch.testing.assert_close(opt.grad_norm, tn, rtol=1e-6, atol=0)
            worst["grad_norm"] = max(worst["grad_norm"], _rel(opt.grad_norm, tn))
        else:
            assert bool(torch.isnan(opt.grad_norm))
        if it == 0:
            for p, q in zip(ours, ref):
                torch.testing.assert_close(p.detach(), q.detach(), rtol=2e-6, atol=1e-7 * float(q.detach().abs().max()))
                worst["step1"] = max(worst["step1"], float((p - q).abs().max()))
    for p, q in zip(ours, ref):
        amax = float(q.detach().abs().max())
        torch.testing.assert_close(p.detach(), q.detach(), rtol=1e-5, atol=1e-6 * amax)
        worst["step50"] = max(worst["step50"], float((p - q).abs().max()) / amax)
        for k in ("exp_avg", "exp_avg_sq"):
            a, b = opt.state[p][k], topt.state[q][k]
            torch.testing.assert_close(a, b, rtol=1e-5, atol=1e-6 * float(b.abs().max()))
        assert float(opt.state[p]["step"]) == 50.0 and opt.state[p]["step"].is_cuda
    if max_norm is not None and max_norm < 10:
        assert float(tn) > max_norm                                      # the clipping was active
    print(f"\n[{name}] max |diff| after 1 step {worst['step1']:.3e}; after 50 steps {worst['step50']:.3e} of max|p|; "
          f"grad_norm rel {worst['grad_norm']:.3e}")


def test_fused_adam_skips_parameters_without_grad(pkg):
    ps = _params(2)
    opt = pkg.FusedAdam(ps, lr=1e-2)
    before = ps[0].detach().clone()
    for p, g in zip(ps[1:], _grads(5, ps[1:], 1e-2)):
        p.grad = g
    v = ps[1]._version
    opt.step()
    assert torch.equal(ps[0].detach(), before) and ps[0] not in opt.state
    assert float(opt.state[ps[1]]["step"]) == 1.0 and ps[1]._version > v


def _run(pkg, seed, steps=10):
    ps = _params(seed)
    opt = pkg.FusedAdamW(ps, lr=1e-2, max_grad_norm=1.0)
    norms = []
    for it in range(steps):
        for p, g in zip(ps, _grads(200 + it, ps, 1e-1)):
            p.grad = g
        opt.step()
        norms.append(opt.grad_norm.clone())
    return ps, opt, torch.stack(norms)


def test_fused_adam_is_bitwise_deterministic(pkg):
    a, oa, na = _run(pkg, 3)
    b, ob, nb = _run(pkg, 3)
    assert torch.equal(na, nb)
    for p, q in zip(a, b):
        assert torch.equal(p, q)
        assert torch.equal(oa.state[p]["exp_avg"], ob.state[q]["exp_avg"])
        assert torch.equal(oa.state[p]["exp_avg_sq"], ob.state[q]["exp_avg_sq"])


def _lr(k):
    return 1e-2 * 0.8 ** k                                               # a schedule: lr changes between steps


def _steps(opt, ps, k0, k1):
    for k in range(k0, k1):
        for g in opt.param_groups:
            g["lr"] = _lr(k)
        for p, g in zip(ps, _grads(300 + k, ps, 1e-2)):
            p.grad = g
        opt.step()


@pytest.mark.parametrize("direction", ["torch_to_fused", "fused_to_torch"])
def test_state_dict_round_trips_with_torch_adam(pkg, direction):
    ref = _params(4)
    topt = torch.optim.Adam(ref, lr=_lr(0), weight_decay=1e-3, foreach=False)
    _steps(topt, ref, 0, 10)
    ps = _params(4)
    first = torch.optim.Adam(ps, lr=_lr(0), weight_decay=1e-3, foreach=False) if direction == "torch_to_fused" \
        else pkg.FusedAdam(ps, lr=_lr(0), weight_decay=1e-3)
    _steps(first, ps, 0, 5)
    second = pkg.FusedAdam(ps, lr=_lr(0), weight_decay=1e-3) if direction == "torch_to_fused" \
        else torch.optim.Adam(ps, lr=_lr(0), weight_decay=1e-3, foreach=False)
    second.load_state_dict(first.state_dict())
    if direction == "torch_to_fused":
        for p in ps:
            assert second.state[p]["step"].is_cuda and float(second.state[p]["step"]) == 5.0
        assert all(g["capturable"] for g in second.param_groups)
    _steps(second, ps, 5, 10)
    for p, q in zip(ps, ref):
        torch.testing.assert_close(p.detach(), q.detach(), rtol=1e-5, atol=1e-6 * float(q.abs().max()))
        st = second.state[p]
        torch.testing.assert_close(st["exp_avg"], topt.state[q]["exp_avg"], rtol=1e-5,
                                   atol=1e-6 * float(topt.state[q]["exp_avg"].abs().max()))
        assert float(st["step"]) == 10.0


def _small_model(pkg, kg, seed=1):
    torch.manual_seed(seed)
    return pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.0, decoder_dropout=0.0).to(DEV)


def _batches(kg, n):
    from primekg_rgcn_linkprediction_b200 import synth
    return [[t.to(DEV) for t in synth.link_batch(kg, 256, seed=10 + i)] for i in range(n)]


def test_graphed_step_with_fused_optimizer_matches_torch(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=5)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = _batches(kg, 4)
    ma, mb = _small_model(pkg, kg), _small_model(pkg, kg)
    ma.train(); mb.train()
    opt_a = pkg.FusedAdam(ma.parameters(), lr=1e-2, max_grad_norm=1.0)
    opt_b = torch.optim.Adam(mb.parameters(), lr=1e-2, foreach=False)
    before = {k: p.detach().clone() for k, p in ma.named_parameters()}
    step_a = pkg.GraphedTrainStep(ma, ei, et, batch_size=512, optimizer=opt_a)
    torch.cuda.synchronize()
    for k, p in ma.named_parameters():                                   # construction moved nothing
        assert torch.equal(p.detach(), before[k]), k
        st = opt_a.state[p]
        assert float(st["step"]) == 0 and not st["exp_avg"].any() and not st["exp_avg_sq"].any(), k
    step_b = pkg.GraphedTrainStep(mb, ei, et, batch_size=512)
    sch_a = torch.optim.lr_scheduler.ExponentialLR(opt_a, 0.9)
    sch_b = torch.optim.lr_scheduler.ExponentialLR(opt_b, 0.9)
    params_b = list(mb.parameters())
    losses = []
    for it in range(20):
        b = batches[it % 4]
        la = float(step_a(*b))
        lb = float(step_b(*b))
        torch.nn.utils.clip_grad_norm_(params_b, 1.0, foreach=False)
        opt_b.step()
        assert abs(la - lb) <= 1e-4 * abs(lb), (it, la, lb)
        assert float(step_a.grad_norm) > 0
        losses.append(la)
        sch_a.step(); sch_b.step()                                         # lr changes after capture, every replay
    # the two runs differ in the last bits from the first update on; Adam divides by sqrt(v), so an entry whose gradient
    # sits at rounding-noise level may step either way: rtol 1e-3 on the whole tensor (relative Frobenius), and every
    # entry within 1 % of the tensor's scale (the bar of test_gpu_reference_calls.py after its Adam steps)
    for (k, p), q in zip(ma.named_parameters(), params_b):
        p, q = p.detach(), q.detach()
        assert float((p - q).norm() / q.norm()) < 1e-3, k
        torch.testing.assert_close(p, q, rtol=1e-3, atol=1e-2 * float(q.abs().max()), msg=lambda s: f"{k}: {s}")
    assert sum(losses[-4:]) < sum(losses[:4])                              # the loss falls
    # lr = 0 set after capture: the next replay updates the moments but not the parameters
    for g in opt_a.param_groups:
        g["lr"] = 0.0
    snap = [p.detach().clone() for p in ma.parameters()]
    m_before = [opt_a.state[p]["exp_avg"].clone() for p in ma.parameters()]
    step_a(*batches[0])
    torch.cuda.synchronize()
    assert all(torch.equal(p.detach(), s) for p, s in zip(ma.parameters(), snap))
    assert any(not torch.equal(opt_a.state[p]["exp_avg"], m) for p, m in zip(ma.parameters(), m_before))
    assert all(float(opt_a.state[p]["step"]) == 21 for p in ma.parameters())


def test_eager_fused_adam_with_autograph_tracks_torch(pkg):
    """The unmodified loop: model(...) (captured by autograph after three calls) + backward + zero_grad + step."""
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=6)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    batches = _batches(kg, 3)
    ma, mb = _small_model(pkg, kg, 2), _small_model(pkg, kg, 2)
    ma.train(); mb.train()
    opt_a = pkg.FusedAdam(ma.parameters(), lr=1e-2)
    opt_b = torch.optim.Adam(mb.parameters(), lr=1e-2)
    for it in range(10):
        b = batches[it % 3]
        for m, opt in ((ma, opt_a), (mb, opt_b)):
            opt.zero_grad()
            loss = F.binary_cross_entropy_with_logits(m(ei, et, b[0], b[1], b[2]), b[3])
            loss.backward()
            opt.step()
    for (k, p), (_, q) in zip(ma.named_parameters(), mb.named_parameters()):
        torch.testing.assert_close(p.detach(), q.detach(), rtol=2e-2, atol=1e-2 * float(q.abs().max()),
                                   msg=lambda s: f"{k}: {s}")


def test_eager_step_invalidates_eval_cache(pkg):
    from primekg_rgcn_linkprediction_b200 import synth
    kg = synth.primekg_subgraph(20_000, seed=7)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    m = _small_model(pkg, kg, 3)
    opt = pkg.FusedAdam(m.parameters(), lr=1e-2)
    m.eval()
    with torch.no_grad():
        cached = m.encoder(ei, et).clone()
    for p in m.parameters():
        p.grad = torch.randn_like(p) * 1e-2
    opt.step()
    with torch.no_grad():
        after = m.encoder(ei, et).clone()
        m.encoder.invalidate_eval_cache()
        fresh = m.encoder(ei, et)
    assert not torch.equal(after, cached)
    assert torch.equal(after, fresh)


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted(e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                  and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())


@pytest.mark.parametrize("clip", [1.0, None])
def test_graphed_step_adds_exactly_the_optimizer_kernels(pkg, clip):
    from primekg_rgcn_linkprediction_b200 import _lib, synth
    lib = _lib.load()
    kg = synth.primekg_subgraph(20_000, seed=8)
    ei, et = kg.edge_index.to(DEV), kg.edge_type.to(DEV)
    b = _batches(kg, 1)[0]
    m = _small_model(pkg, kg, 4)
    m.train()
    pkg.GraphedTrainStep(m, ei, et, batch_size=512)                      # one-time work (graph build, plans) first
    for p in m.parameters():
        p.grad = None
    n0 = lib.rgcn_launch_count()
    plain = pkg.GraphedTrainStep(m, ei, et, batch_size=512)
    n_plain = lib.rgcn_launch_count() - n0
    plain.load_batch(*b)
    k_plain = _kernel_names(plain)
    del plain
    for p in m.parameters():
        p.grad = None
    opt = pkg.FusedAdam(m.parameters(), lr=1e-3, max_grad_norm=clip)
    n0 = lib.rgcn_launch_count()
    step = pkg.GraphedTrainStep(m, ei, et, batch_size=512, optimizer=opt)
    n_opt = lib.rgcn_launch_count() - n0
    n_adam = 2 if clip is not None else 1
    assert n_opt == n_plain + n_adam                                       # only the captured pass launches it
    n0 = lib.rgcn_launch_count()
    step.load_batch(*b)
    k_opt = _kernel_names(step)
    assert lib.rgcn_launch_count() == n0                                   # a replay launches nothing from the host
    extra = list(k_opt)
    for k in k_plain:
        extra.remove(k)
    assert len(extra) == n_adam and all("adam_" in k for k in extra), extra


def _dp_worker(rank, port, ret):
    import sys
    from conftest import ROOT
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=2, device_id=dev)
    try:
        import primekg_rgcn_linkprediction_b200 as pkg
        from primekg_rgcn_linkprediction_b200 import synth
        kg = synth.primekg_subgraph(40_000, seed=3)
        ei, et = kg.edge_index.to(dev), kg.edge_type.to(dev)
        torch.manual_seed(1)
        model = pkg.DrugDiseaseModel(kg.num_nodes, kg.num_relations, 64, 128, dropout=0.0, decoder_dropout=0.0).to(dev)
        model.train()
        opt = pkg.FusedAdam(model.parameters(), lr=1e-2, max_grad_norm=1.0)
        step = pkg.GraphedTrainStep(model, ei, et, batch_size=512, flat_grads="arena", allreduce="peer", optimizer=opt)
        for it in range(10):
            b = [t.to(dev) for t in synth.link_batch(kg, 256, seed=100 * rank + it)]       # different data per rank
            step(*b)
        step.peer_ar.check()
        flat = torch.cat([p.detach().reshape(-1) for p in model.parameters()])
        both = [torch.empty_like(flat) for _ in range(2)]
        dist.all_gather(both, flat)
        ret[rank] = bool(torch.equal(both[0], both[1])) and all(float(opt.state[p]["step"]) == 10
                                                                  for p in model.parameters())
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_allreduce_with_optimizer_keeps_replicas_identical_two_gpus(lib_built):
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.get_context("spawn").Manager().dict()
    mp.spawn(_dp_worker, args=(port, ret), nprocs=2, join=True)
    assert ret.get(0) is True and ret.get(1) is True
