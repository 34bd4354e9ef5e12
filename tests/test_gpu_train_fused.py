"""-m gpu: training-mode BatchNorm on the fused kernel (spsnet_b200/train_fused.py, SURVEY.md section 8(f) rank 4).

  * the statistics pass of spsk_sa_mma_forward against a float64 evaluation of the same chain (every launch shape: resident
    narrow / split, ring, two epilogue groups, many tiles per CTA, ragged last tile), bit-reproducible;
  * a set-abstraction module in train(): fused vs the reference composition of the same module (SPSK_TRAIN_FUSED=0) -- pooled
    features within 1e-3, running statistics, and -- with the same upstream gradient -- every gradient;
  * the drop-in module in train() against recorded outputs of the same module and batch (tests/helpers.py::Recorded) and,
    where oracle/_ref is installed, against the UNMODIFIED reference module + its CUDA ops in train():
    forward, running statistics of every BatchNorm layer, parameter gradients
    (reference pointnet2_modules.py:203-211, 429-445; pointnet2_utils.py:184-222 for the grouping backward)."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

from helpers import assert_close, rel_err  # noqa: E402
from spsnet_b200 import scenes  # noqa: E402


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.fixture(autouse=True)
def _fp32_truth():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


# (name, c_feat, widths, nsample, B, N, M)
STAT_CASES = [
    ("narrow_split", 1, [16, 16, 32], 16, 2, 2048, 512),         # resident, split arithmetic, 4 CTAs per SM
    ("narrow_ragged", 1, [32, 32, 64], 16, 1, 1000, 100),        # 1600 rows: 12 full tiles + half a tile
    ("plain_mid", 64, [64, 64, 128], 32, 2, 1024, 256),          # plain fp16 operands, resident
    ("plain_1layer", 64, [96], 16, 2, 1024, 256),                # statistics of the FIRST conv (a one-layer chain)
    ("ring_two_groups", 256, [256, 512, 1024], 32, 4, 2048, 1024),   # streaming ring, G = 2, 8 cout chunks, ~7 tiles per CTA
    ("xyz_only", 0, [16, 32], 8, 2, 512, 128),
]


@pytest.mark.parametrize("name,c_feat,widths,ns,B,N,M", STAT_CASES, ids=[c[0] for c in STAT_CASES])
def test_statistics_pass_vs_float64(name, c_feat, widths, ns, B, N, M):
    from spsnet_b200 import pointnet2_utils as pu

    torch.manual_seed(3)
    xyz = dev(scenes.make_batch(21, B, N)[:, :, :3])
    sel = pu.furthest_point_sample(xyz, M)
    new_xyz = pu.gather_rows(xyz, sel)
    feats = (torch.randn(B, c_feat, N, device="cuda") * 0.7 + 0.2) if c_feat else None
    idx = pu.ball_query(1.2, ns, xyz, new_xyz)
    cin = c_feat + 3
    chain = []
    for l, cout in enumerate(widths):
        wt = torch.randn(cin, cout, device="cuda") / cin ** 0.5
        last = l == len(widths) - 1
        bias = torch.zeros(cout, device="cuda") if last else torch.randn(cout, device="cuda") * 0.2
        chain.append((wt, bias, True))
        cin = cout
    pk = pu.MmaChain(chain, c_feat, True, pair=False)
    assert pk.ok
    nparts = pu.sa_mma_stats_parts(idx, N, pk)
    twin = pu.make_twin(feats, (c_feat + 7) // 8 * 8) if (c_feat and not pk.split) else None

    def run():
        # one guard slice on either side of the buffer: the kernel must write exactly `nparts` slices
        guarded = torch.full((nparts + 2, pk.cpad[-1], 2), -777.0, dtype=torch.float64, device="cuda")
        parts = guarded[1:nparts + 1]
        parts.zero_()
        pu.sa_mma_forward(xyz=xyz, new_xyz=new_xyz, idx=idx, chain=pk, twin=twin, features=feats if pk.split else None, stats=parts)
        assert bool((guarded[0] == -777.0).all()) and bool((guarded[-1] == -777.0).all()), "statistics pass wrote outside its slices"
        return parts.clone()

    parts = run()
    assert torch.equal(parts, run())                                   # per-thread cells, no atomics: reproducible bit for bit
    sums = parts.sum(0)
    assert float(sums[widths[-1]:].abs().max() if pk.cpad[-1] > widths[-1] else 0.0) == 0.0   # padded couts: exactly zero
    # float64 truth from the reference composition of the grouped tensor
    g = pu._group(xyz, new_xyz, feats, idx, True).double()            # (B, 3 + C, M, ns)
    rows = g.permute(0, 2, 3, 1).reshape(-1, g.shape[1])
    for l, (wt, bias, _) in enumerate(chain):
        z = rows @ wt.double()
        rows = torch.relu(z + bias.double())
    count = B * M * ns
    mean_w, var_w = z.mean(0), z.var(0, unbiased=False)
    mean = sums[:widths[-1], 0] / count
    var = sums[:widths[-1], 1] / count - mean * mean
    std = var_w.sqrt()
    e_mean = float(((mean - mean_w).abs() / (std + mean_w.abs() + 1e-12)).max())
    e_var = float(((var - var_w).abs() / (var_w + 1e-12)).max())
    print(f"[stats] {name}: parts={nparts} split={pk.split} ctas/SM={pk.ctas_per_sm} resident={pk.resident} mean err {e_mean:.2e} var err {e_var:.2e}")
    assert e_mean <= 1e-3 and e_var <= 2e-3


PACK_CASES = [(1, [16, 16, 32]), (1, [32, 32, 64]), (64, [64, 96, 128]), (128, [128, 256, 256]), (256, [256, 512, 1024]), (0, [16, 32]),
              (5, [17, 33]), (20, [40])]


@pytest.mark.parametrize("c_feat,widths", PACK_CASES, ids=[f"c{c}-" + "x".join(map(str, w)) for c, w in PACK_CASES])
def test_pack_layer_kernel_equals_host_packing(c_feat, widths):
    """spsk_sa_pack_layer (one launch per layer, from the Conv2d weight [x BN scale]) writes byte for byte what pu.MmaChain packs
    with torch ops: layer-0 permutation, hi/lo split, ragged k tiles and cout chunks, zero padding."""
    from spsnet_b200 import pointnet2_utils as pu
    from spsnet_b200 import train_fused as tf

    torch.manual_seed(1)
    cin = c_feat + 3
    convs, scales = [], []
    for co in widths:
        convs.append(torch.randn(co, cin, device="cuda") / cin ** 0.5)
        scales.append(torch.rand(co, device="cuda") + 0.5)
        cin = co
    split = c_feat <= 8 and all(tf._ceil(co, 16) <= 64 for co in widths[:-1])
    plan = tf.TrainPlan([tuple(w.shape) for w in convs], c_feat, True, split, "cuda")
    assert plan.ok
    for use_scale in (False, True):
        plan.wbuf.fill_(0xAB)                                                # stale bytes: padding must be WRITTEN, not assumed
        chain = []
        for l, w in enumerate(convs):
            sc = scales[l] if use_scale else None
            plan.pack(l, w, sc, last=l == len(convs) - 1)
            chain.append(((w * sc[:, None] if use_scale else w).t().contiguous(), torch.zeros(w.shape[0], device="cuda"), True))
        want = pu.MmaChain(chain, c_feat, True, split=split, pair=False)
        assert want.split == split
        got = plan.wbuf[:want.wtiles.numel() * 2].view(torch.float16)
        assert torch.equal(got.view(torch.int16), want.wtiles.view(torch.int16)), f"scale={use_scale}"
        tail = plan.wbuf[want.wtiles.numel() * 2:]
        assert tail.numel() == 0 or bool((tail == 0xAB).all()), "the pack kernel wrote past the chain's tiles"


@pytest.mark.parametrize("momentum", [0.1, None])
def test_reduce_and_finalize_kernels_equal_host_algebra(momentum):
    from spsnet_b200 import train_fused as tf

    torch.manual_seed(2)
    c, cpad, nparts, count = 96, 128, 37, 37 * 128 * 5
    z = torch.randn(nparts, 128 * 5, c, device="cuda", dtype=torch.float64) * 1.7 + 0.4
    parts = torch.zeros(nparts, cpad, 2, device="cuda", dtype=torch.float64)
    parts[:, :c, 0] = z.sum(1)
    parts[:, :c, 1] = (z * z).sum(1)
    bn_k, bn_t = nn.BatchNorm2d(c, momentum=momentum).cuda().train(), None
    bn_k.weight.data.uniform_(0.5, 1.5)
    bn_k.bias.data.uniform_(-0.3, 0.3)
    bn_k.running_mean.normal_()
    bn_k.running_var.uniform_(0.5, 2.0)
    bn_t = copy.deepcopy(bn_k)
    w = torch.randn(c, 40, device="cuda")
    plan = tf.TrainPlan([(c, 40)], 37, True, False, "cuda")
    for step in range(2):
        plan.finalize(0, parts, count, bn_k, bn_k.weight.detach(), bn_k.bias.detach(), None)
        mean, var, total = tf.bn_moments(parts.sum(0)[:c], count)
        tf.bn_update_running(bn_t, mean, var, total)
        wt, bias = tf.bn_fold(w, bn_t.weight.detach(), bn_t.bias.detach(), mean, var, bn_t.eps)
        assert torch.allclose(plan.bbuf[:c], bias, rtol=1e-5, atol=1e-6)
        assert torch.allclose((w * plan.scale[0][:, None]).t(), wt, rtol=1e-5, atol=1e-6)
        assert float(plan.bbuf[c:].abs().max()) == 0.0
    assert torch.allclose(bn_k.running_mean, bn_t.running_mean, rtol=1e-5, atol=1e-6)
    assert torch.allclose(bn_k.running_var, bn_t.running_var, rtol=1e-5, atol=1e-6)
    assert int(bn_k.num_batches_tracked) == int(bn_t.num_batches_tracked) == 2
    assert float(plan.sums[0][-1]) == float(count)


def test_kernel_and_torch_host_paths_agree(monkeypatch):
    """SPSK_TRAIN_PACK=torch (host algebra in torch ops, folded in fp64) and the default device-side kernels give the same
    training forward up to the fp32 rounding of the fold."""
    from spsnet_b200 import pointnet2_utils as pu

    outs, stats = [], []
    for mode in ("kernel", "torch"):
        monkeypatch.setenv("SPSK_TRAIN_PACK", mode)
        m = _msg_module("l1", seed=6)
        xyz = dev(scenes.make_batch(35, 2, 1024)[:, :, :3])
        new_xyz = pu.gather_rows(xyz, pu.furthest_point_sample(xyz, 256))
        torch.manual_seed(8)
        feats = torch.randn(2, 64, 1024, device="cuda")
        out, _ = m._msg(xyz, new_xyz, feats)
        outs.append(out.detach())
        stats.append([(b.running_mean.clone(), b.running_var.clone()) for b in m.modules() if isinstance(b, nn.BatchNorm2d)])
    assert rel_err(outs[0].cpu().numpy(), outs[1].cpu().numpy()) <= 2e-5
    for (m0, v0), (m1, v1) in zip(*stats):
        assert torch.allclose(m0, m1, rtol=1e-5, atol=1e-7) and torch.allclose(v0, v1, rtol=1e-5, atol=1e-7)


MSG_CASES = {
    # KITTI layer 0 (split chains), layer 1 (plain, resident), layer 2 scale 2 widths (ring) -- small point counts
    "l0": dict(cin=1, radii=[0.2, 0.8], nsamples=[16, 32], mlps=[[1, 16, 16, 32], [1, 32, 32, 64]], n=2048, m=512),
    "l1": dict(cin=64, radii=[0.8, 1.6], nsamples=[16, 32], mlps=[[64, 64, 64, 128], [64, 64, 96, 128]], n=1024, m=256),
    "l2": dict(cin=128, radii=[1.6, 4.8], nsamples=[16, 32], mlps=[[128, 128, 128, 256], [128, 128, 256, 256]], n=512, m=128),
    "dil": dict(cin=5, radii=[0.8, 1.6], nsamples=[16, 32], mlps=[[5, 17, 33], [5, 24, 40]], n=700, m=100, dilated=True),
}


def _msg_module(kind, seed=0):
    from spsnet_b200 import pointnet2_modules as pm

    c = MSG_CASES[kind]
    torch.manual_seed(seed)
    if c.get("dilated"):
        m = pm.PointnetSAModuleMSG_WithSampling(npoint_list=[c["m"]], sample_range_list=[-1], sample_type_list=["D-FPS"], radii=c["radii"],
                                                nsamples=c["nsamples"], mlps=copy.deepcopy(c["mlps"]), dilated_group=True,
                                                aggregation_mlp=None, confidence_mlp=None, num_class=3)
    else:
        m = pm.PointnetSAModuleMSG(npoint=c["m"], radii=c["radii"], nsamples=c["nsamples"], mlps=copy.deepcopy(c["mlps"]), use_xyz=True)
    for mod in m.modules():
        if isinstance(mod, nn.BatchNorm2d):
            mod.weight.data.uniform_(0.5, 1.5)
            mod.bias.data.uniform_(-0.2, 0.2)
    return m.cuda().train()


@pytest.mark.parametrize("kind", list(MSG_CASES))
def test_msg_train_fused_vs_composition(kind, monkeypatch):
    """Same module, same inputs, same upstream gradient: fused statistics + pooled pass + recompute backward against the
    reference composition with torch BatchNorm2d in train()."""
    from spsnet_b200 import pointnet2_utils as pu

    c = MSG_CASES[kind]
    B = 2
    fused = _msg_module(kind, seed=4)
    comp = copy.deepcopy(fused)
    xyz = dev(scenes.make_batch(33, B, c["n"])[:, :, :3])
    new_xyz0 = pu.gather_rows(xyz, pu.furthest_point_sample(xyz, c["m"]))
    feats0 = torch.randn(B, c["cin"], c["n"], device="cuda")
    outs, grads, stats = [], [], []
    for mod, flag in ((fused, "1"), (comp, "0")):
        monkeypatch.setenv("SPSK_TRAIN_FUSED", flag)
        feats = feats0.clone().requires_grad_(True)
        new_xyz = new_xyz0.clone().requires_grad_(True)
        for step in range(2):                                      # two steps: running statistics chain through the momentum update
            out, _ = mod._msg(xyz, new_xyz, feats)
        torch.manual_seed(9)
        gout = torch.randn_like(out)
        params = [p for p in mod.parameters()]
        g = torch.autograd.grad(out, [feats, new_xyz] + params, gout)
        outs.append(out.detach())
        grads.append(g)
        stats.append([(b.running_mean.clone(), b.running_var.clone(), int(b.num_batches_tracked)) for b in mod.modules() if isinstance(b, nn.BatchNorm2d)])
    assert outs[0].shape == outs[1].shape
    assert_close(outs[0].cpu().numpy(), outs[1].cpu().numpy(), what=f"{kind} pooled features, train()")
    for (m0, v0, n0), (m1, v1, n1) in zip(*stats):
        assert n0 == n1 == 2
        assert rel_err(m0.cpu().numpy(), m1.cpu().numpy()) <= 1e-3
        assert rel_err(v0.cpu().numpy(), v1.cpu().numpy()) <= 2e-3
    names = ["features", "new_xyz"] + [n for n, _ in fused.named_parameters()]
    for n, a, b in zip(names, *grads):
        e = rel_err(a.cpu().numpy(), b.cpu().numpy())
        assert e <= 2e-4, f"{kind}: grad {n} relative error {e:.2e}"


def test_fused_training_is_the_path_taken(monkeypatch):
    """train() really runs the statistics kernel (and the composition is used when it is switched off)."""
    from spsnet_b200 import pointnet2_utils as pu
    from spsnet_b200._lib import lib

    m = _msg_module("l1", seed=1)
    xyz = dev(scenes.make_batch(34, 2, 1024)[:, :, :3])
    new_xyz = pu.gather_rows(xyz, pu.furthest_point_sample(xyz, 256))
    feats = torch.randn(2, 64, 1024, device="cuda", requires_grad=True)
    calls = []
    real = pu.sa_mma_forward
    monkeypatch.setattr(pu, "sa_mma_forward", lambda **kw: (calls.append("stats" if kw.get("stats") is not None else "pool"), real(**kw))[1])
    out, _ = m._msg(xyz, new_xyz, feats)
    assert calls == ["stats", "stats", "stats", "pool"] * 2 and out.requires_grad
    calls.clear()
    monkeypatch.setenv("SPSK_TRAIN_FUSED", "0")
    m._msg(xyz, new_xyz, feats)
    assert calls == []
    assert lib.spsk_abi_version() >= 4


REF_KINDS = {
    "l0": dict(npoint_list=[512], sample_type_list=["D-FPS"], radii=[0.2, 0.8], nsamples=[16, 32],
               mlps=[[1, 16, 16, 32], [1, 32, 32, 64]], aggregation_mlp=[64], confidence_mlp=None, cin=1, n=2048),
    "l1": dict(npoint_list=[256], sample_type_list=["D-FPS"], radii=[0.8, 1.6], nsamples=[16, 32],
               mlps=[[64, 64, 64, 128], [64, 64, 96, 128]], aggregation_mlp=[128], confidence_mlp=[128], cin=64, n=1024),
}


@pytest.mark.parametrize("kind", list(REF_KINDS))
def test_sa_module_train_vs_reference_module_train(ref_ops, recorded, kind):
    """The drop-in module in train() against the recorded outputs of the same module and batch in train()
    (tests/helpers.py::Recorded) and, where oracle/_ref is installed, against the unmodified reference module + CUDA ops in
    train(): same state_dict, same batch -- sampled indices bit-exact, features / logits within 1e-3 / 3e-3, every
    BatchNorm's running statistics, and the parameter gradients of a fixed linear loss."""
    from spsnet_b200 import pointnet2_modules as pm

    kw = copy.deepcopy(REF_KINDS[kind])
    cin, n = kw.pop("cin"), kw.pop("n")
    torch.manual_seed(2)
    ours = pm.PointnetSAModuleMSG_WithSampling(sample_range_list=[-1], num_class=3, **copy.deepcopy(kw)).cuda().train()
    for mod in ours.modules():
        if isinstance(mod, (nn.BatchNorm1d, nn.BatchNorm2d)):
            mod.weight.data.uniform_(0.5, 1.5)
            mod.bias.data.uniform_(-0.2, 0.2)
    mods = [ours]
    if ref_ops is not None:
        ref = ref_ops.modules.PointnetSAModuleMSG_WithSampling(sample_range_list=[-1], num_class=3, **copy.deepcopy(kw)).cuda().train()
        ref.load_state_dict(ours.state_dict())
        mods += [ref, copy.deepcopy(ref)]    # the last one runs as shipped: its convolutions in TF32
    B = 2
    xyz = dev(scenes.make_batch(61, B, n)[:, :, :3])
    feats = torch.randn(B, cin, n, device="cuda")
    res = []
    tf32 = torch.backends.cudnn.allow_tf32
    try:
        for i, mod in enumerate(mods):
            torch.backends.cudnn.allow_tf32 = i == 2
            out = mod(xyz, feats.clone(), None)
            torch.manual_seed(13)
            loss = (out[1] * torch.randn_like(out[1])).sum()
            if out[2] is not None:
                loss = loss + (out[2] * torch.randn_like(out[2])).sum()
            mod.zero_grad()
            loss.backward()
            res.append(out)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    out = res[0]
    recorded.exact("idx", out[3])
    recorded.exact("new_xyz", out[0])
    recorded.close("new_features", out[1])
    # Class logits in train(): two batch-normalised Conv1d layers (aggregation, confidence) renormalise every channel by its
    # BATCH standard deviation, which magnifies the ~4e-4 deviation of the pooled features.  Bar for the logits in training
    # mode: 3e-3 (the 1e-3 bar is the inference bar, tests/test_gpu_modules.py, where these layers run on hi + lo arithmetic
    # with fixed statistics).
    if out[2] is not None:
        recorded.close("cls", out[2], 3e-3)
    for k, v in ours.state_dict().items():
        if k.endswith("running_mean") or k.endswith("running_var"):
            recorded.close(k, v, 2e-3, k=128)
        if k.endswith("num_batches_tracked"):
            assert int(v) == 1
    # Parameter gradients.  The backward of the fused path differentiates the fp32 reference function at the same inputs
    # (test_msg_train_fused_vs_composition: <= 2e-4 for the same upstream gradient); end to end the upstream gradient itself
    # moves with the ~1e-3 forward deviation, through two batch-normalised Conv1d layers and this random-projection loss.  The
    # reference's own stock (TF32) run moves by the same amount (scripts/diag_train_grads.py, profiles/r02_diag_train_grads.txt),
    # so the bar is: the split-arithmetic chains (l0) match tightly, and the fp16-operand chains stay within 0.25 and, against
    # the live reference, within 3x of what the reference's shipped configuration does against its own fp32 run.
    worst = 0.0
    for name, p in ours.named_parameters():
        assert p.grad is not None, name
        worst = max(worst, recorded.err(name + ".grad", p.grad, k=128))
    print(f"[train vs recorded] {kind}: worst parameter-gradient relative error {worst:.2e}")
    assert worst <= (1e-4 if kind == "l0" else 0.25)
    if ref_ops is None:
        return
    ref, stock = mods[1], mods[2]
    np.testing.assert_array_equal(res[0][3].cpu().numpy(), res[1][3].cpu().numpy())
    np.testing.assert_array_equal(res[0][0].detach().cpu().numpy(), res[1][0].detach().cpu().numpy())
    assert_close(res[0][1].detach().cpu().numpy(), res[1][1].detach().cpu().numpy(), what=f"{kind} new_features, train()")
    if res[1][2] is not None:
        e = rel_err(res[0][2].detach().cpu().numpy(), res[1][2].detach().cpu().numpy())
        e_stock = rel_err(res[2][2].detach().cpu().numpy(), res[1][2].detach().cpu().numpy())
        print(f"[train vs reference] {kind}: logits ours {e:.2e} / stock-TF32 {e_stock:.2e}")
        assert e <= 3e-3, f"{kind} cls logits, train(): relative error {e:.3e} > 3e-3"
    sd_o, sd_r = ours.state_dict(), ref.state_dict()
    for k in sd_o:
        if k.endswith("running_mean") or k.endswith("running_var"):
            e = rel_err(sd_o[k].cpu().numpy(), sd_r[k].cpu().numpy())
            assert e <= 2e-3, f"{kind}: {k} relative error {e:.2e}"
        if k.endswith("num_batches_tracked"):
            assert int(sd_o[k]) == int(sd_r[k]) == 1
    worst = worst_stock = 0.0
    for (name, p), (_, q), (_, t) in zip(ours.named_parameters(), ref.named_parameters(), stock.named_parameters()):
        assert p.grad is not None and q.grad is not None, name
        worst = max(worst, rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()))
        worst_stock = max(worst_stock, rel_err(t.grad.cpu().numpy(), q.grad.cpu().numpy()))
    print(f"[train vs reference] {kind}: worst parameter-gradient relative error ours {worst:.2e} / stock-TF32 {worst_stock:.2e}")
    if kind == "l0":
        assert worst <= 1e-4
    else:
        assert worst <= 0.25 and worst <= 3.0 * worst_stock


def test_composition_in_train_mode_is_the_reference_exactly(ref_ops, recorded, monkeypatch):
    """SPSK_TRAIN_FUSED=0: the drop-in module in train() on the op-by-op composition reproduces the forward, running
    statistics and parameter gradients of the same module and batch to fp32 rounding: the recorded ones
    (tests/helpers.py::Recorded) and, where oracle/_ref is installed, the reference module's (same torch layers over
    bit-exact CUDA ops)."""
    from spsnet_b200 import pointnet2_modules as pm

    monkeypatch.setenv("SPSK_TRAIN_FUSED", "0")
    kw = copy.deepcopy(REF_KINDS["l1"])
    cin, n = kw.pop("cin"), kw.pop("n")
    torch.manual_seed(3)
    ours = pm.PointnetSAModuleMSG_WithSampling(sample_range_list=[-1], num_class=3, **copy.deepcopy(kw)).cuda().train()
    mods = [ours]
    if ref_ops is not None:
        ref = ref_ops.modules.PointnetSAModuleMSG_WithSampling(sample_range_list=[-1], num_class=3, **copy.deepcopy(kw)).cuda().train()
        ref.load_state_dict(ours.state_dict())
        mods.append(ref)
    xyz = dev(scenes.make_batch(62, 2, n)[:, :, :3])
    feats = torch.randn(2, cin, n, device="cuda")
    for mod in mods:
        out = mod(xyz, feats.clone(), None)
        torch.manual_seed(14)
        ((out[1] * torch.randn_like(out[1])).sum() + (out[2] * torch.randn_like(out[2])).sum()).backward()
        mod._out = out
    recorded.close("new_features", ours._out[1], 1e-5)
    for name, p in ours.named_parameters():
        recorded.close(name + ".grad", p.grad, 1e-4, k=128)
    for k, v in ours.state_dict().items():
        if "running" in k:
            recorded.close(k, v, 1e-5, k=128)
    if ref_ops is None:
        return
    assert rel_err(ours._out[1].detach().cpu().numpy(), ref._out[1].detach().cpu().numpy()) <= 1e-5
    for (name, p), (_, q) in zip(ours.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad.cpu().numpy(), q.grad.cpu().numpy()) <= 1e-4, name
    for (k, a), (_, b) in zip(ours.state_dict().items(), ref.state_dict().items()):
        if "running" in k:
            assert rel_err(a.cpu().numpy(), b.cpu().numpy()) <= 1e-5, k


def test_backbone_training_step_runs_on_the_fused_path(monkeypatch):
    """A whole IA-SSD SA stack in train(): forward + backward + SGD step, finite, every grouped-MLP BatchNorm updated once."""
    from helpers import small_sa_cfg
    from spsnet_b200 import backbone as bb
    from spsnet_b200 import pointnet2_utils as pu

    torch.manual_seed(0)
    net = bb.IASSD_Backbone(small_sa_cfg((512, 128, 64, 32)), num_class=3, input_channels=4).cuda().train()
    calls = []
    real = pu.sa_mma_forward
    monkeypatch.setattr(pu, "sa_mma_forward", lambda **kw: (calls.append(kw.get("stats") is not None), real(**kw))[1])
    B, N = 2, 2048
    pts = dev(scenes.to_points(scenes.make_batch(81, B, N)))
    opt = torch.optim.SGD(net.parameters(), lr=1e-3)
    out = net({"batch_size": B, "points": pts})
    loss = out["centers_features"].square().mean() + out["ctr_offsets"][:, 1:].square().mean()
    loss.backward()
    opt.step()
    assert torch.isfinite(loss)
    assert sum(calls) == 4 * 2 * 3 and len(calls) - sum(calls) == 4 * 2      # 4 MSG layers x 2 scales x (3 statistics passes + 1 pooled pass)
    n2d = [m for m in net.modules() if isinstance(m, nn.BatchNorm2d)]
    assert n2d and all(int(m.num_batches_tracked) == 1 for m in n2d)
    grads = [p.grad for p in net.parameters() if p.grad is not None]
    assert grads and all(torch.isfinite(g).all() for g in grads)
