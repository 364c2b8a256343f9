"""GPU numerics of the leaf-evaluation pipeline: fused inference plans (library convs/GEMMs + the
engine's stem / heads kernels) against the plain PyTorch fp32 modules in eval mode.
Tolerances: fp32 plan 2e-5 abs on probabilities/values (north_star: Q/priors within 1e-5 relative is
for the TREE given identical net outputs; the net itself is floating point and its plan re-associates
sums); bf16 plans: BF16_BOUNDS below (relative error of every prior above 1e-3, per-row KL, tanh value) against the
fp32 module on bf16-rounded weights."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _randomise_bn(model, seed):
    g = torch.Generator().manual_seed(seed)
    for m in model.modules():
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.BatchNorm1d)):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.3)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.2)


def _rounded_copy(model, dtype):
    """The fp32 module with every conv / linear weight rounded to `dtype` (what a 16-bit plan can represent at best)."""
    import copy
    m = copy.deepcopy(model)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, (torch.nn.Conv2d, torch.nn.Linear)):
                mod.weight.copy_(mod.weight.to(dtype).float())
    return m


def _net_errors(p, v, p_ref, v_ref):
    """max relative error over every prior above 1e-3, largest per-row KL(ref || p), max |v - v_ref|, max abs prior error."""
    big = p_ref > 1e-3
    rel = ((p - p_ref).abs() / p_ref)[big].max().item()
    kl = (p_ref * (torch.log(p_ref.clamp_min(1e-30)) - torch.log(p.clamp_min(1e-30)))).sum(1).max().item()
    return {"rel": rel, "kl": kl, "v": (v - v_ref).abs().max().item(), "abs": (p - p_ref).abs().max().item()}


def _record(name, errs):
    """Achieved errors go to gpurun_out/net_errors.json (scratch) so that the bounds below can be read against them."""
    import json
    import os
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "net_errors.json")
    try:
        os.makedirs(os.path.dirname(path), exist_ok=True)
        d = json.load(open(path)) if os.path.exists(path) else {}
        d[name] = errs
        json.dump(d, open(path, "w"), indent=1, sort_keys=True)
    except OSError:
        pass


# bf16 bounds per net, every one about 3x what the plans achieve on a B200 (profiles/r02_net_errors.md; BatchNorm
# statistics and weights are random here, which makes the nets far more sensitive than trained ones): relative error of
# every prior above 1e-3, per-row KL divergence, tanh value.  A wrong fold of one BatchNorm moves the KL by orders of magnitude.
BF16_BOUNDS = {("simple", 3): {"rel": 1.5e-2, "kl": 1e-5, "v": 8e-3}, ("simple", 5): {"rel": 1.5e-2, "kl": 1e-5, "v": 8e-3},
               ("resnet", 3): {"rel": 1e-1, "kl": 3e-4, "v": 2e-2}, ("resnet", 5): {"rel": 3e-1, "kl": 2.5e-3, "v": 5e-2},
               ("simple", 6): {"rel": 1e-2, "kl": 2.5e-6, "v": 3e-3}, ("simple", 7): {"rel": 1.2e-2, "kl": 2.5e-6, "v": 3.2e-3},
               ("resnet", 7): {"rel": 5e-1, "kl": 8e-3, "v": 1e-4}}
# the plain bf16 module (no fused plan) exponentiates a bf16 log_softmax: looser; for ResNetZero on 7x7 (128 policy outputs
# after 4 blocks with random BatchNorm) the relative bound is about 3x its measured 0.26 (profiles/r02_net_errors.md)
MODULE_BOUNDS = {"rel": 1.5e-1, "kl": 2e-2, "v": 3e-2}
MODULE_BOUNDS_BY_NET = {("resnet", 7): {"rel": 7.5e-1, "kl": 2e-2, "v": 3e-2}}


@pytest.mark.parametrize("net,board,blocks", [("simple", (3, 3), 0), ("simple", (5, 5), 0), ("resnet", (3, 3), 4), ("resnet", (5, 5), 4),
                                              ("resnet", (3, 3), 20), ("resnet", (5, 5), 20), ("simple", (6, 6), 0), ("simple", (7, 7), 0),
                                              ("resnet", (7, 7), 4)])
def test_fused_plans_match_torch_modules(net, board, blocks):
    """fp32 plan: 2e-5 abs against the fp32 module.  bf16 plans: against the fp32 module evaluated on bf16-rounded
    weights -- a relative bound on every prior above 1e-3, a per-row KL bound and an absolute bound on the tanh value
    (BF16_BOUNDS); ResNetZero also at its full depth of 20 blocks (configuration.py:133-155), with the tcgen05 tower
    kernel and with the library convolutions.  On 6x6 and 7x7 (98 and 128 actions: the fourth logit slot of the heads
    kernels) the tower kernel does not apply and the plans run on library convolutions."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine
    from dotsboxesaz_b200.nn import (DeviceEvaluator, FusedResNetZero, FusedSimpleNN, ResNetZero, resnet_zero_parameters)
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.utils.utils import DotDict
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n = 512
    eng = engine.Engine(board, n_games=n, max_nodes=64)
    torch.manual_seed(1)
    if net == "simple":
        model = SimpleNN(board=board)
        plan_cls = FusedSimpleNN
    else:
        model = ResNetZero(DotDict({"nn": {"model_parameters": resnet_zero_parameters(board, nb_blocks=blocks)}}))
        plan_cls = FusedResNetZero
    _randomise_bn(model, 2)
    model = model.cuda().eval()
    # leaves of a real search as inputs
    st = eng.new_states(n)
    plies, _ = eng.random_rollout(st.clone(), seed=3, record_moves=True)
    for ply in range(6):
        legal = eng.valid_moves(st).float()
        mv = torch.multinomial(legal + 1e-9, 1).reshape(-1).int()
        eng.play(st, torch.where(torch.arange(n, device=st.device) % 7 > ply, mv, torch.full_like(mv, -1)))
    x32 = eng.features(st, torch.float32)
    with torch.no_grad():
        logp, v = model(x32)
        logp16, v16 = _rounded_copy(model, torch.bfloat16)(x32)
    refs = {torch.float32: (torch.exp(logp), v.reshape(-1)), torch.bfloat16: (torch.exp(logp16), v16.reshape(-1))}
    tag = "%s-%dx%d-%d" % (net, board[0], board[1], blocks)

    def check(name, dtype):
        torch.cuda.synchronize()
        p_ref, v_ref = refs[dtype]
        assert torch.isfinite(eng.priors).all()
        # the plans' heads kernel normalises in float32; the plain bf16 module exponentiates a bf16 log_softmax
        assert (eng.priors.sum(1) - 1).abs().max() < (1e-3 if name.startswith("plan") else 1e-2)
        errs = _net_errors(eng.priors, eng.values, p_ref, v_ref)
        _record("%s %s" % (tag, name), errs)
        if dtype == torch.float32:
            assert errs["abs"] < 2e-5 and errs["v"] < 2e-5, (tag, name, errs)
        else:
            bounds = BF16_BOUNDS[(net, board[0])] if name.startswith("plan") else MODULE_BOUNDS_BY_NET.get((net, board[0]), MODULE_BOUNDS)
            for k, bound in bounds.items():
                assert abs(errs[k]) < bound, (tag, name, k, errs)

    for dtype in (torch.float32, torch.bfloat16):
        dn = "fp32" if dtype == torch.float32 else "bf16"
        plan = plan_cls(model, eng, dtype=dtype)
        eng.planes.copy_(x32.to(dtype))
        eng.leaf_states.copy_(st)
        plan(eng)
        check("plan " + dn, dtype)
        if dtype != torch.float32:
            assert plan.stem_mma is not None  # the default stem is the tensor-core kernel
            if net == "resnet" and eng.tower_geometry()["ok"]:
                assert plan.tower is not None  # ... and the default tower the tcgen05 kernel (up to 5x5 boxes)
                plan_lib = plan_cls(model, eng, dtype=dtype, use_tower=False)
                assert plan_lib.tower is None
                plan_lib(eng)
                check("plan bf16, library convolutions", dtype)
            if blocks <= 4:  # the library-conv0 and the CUDA-core-stem variants of the same plan must agree as well
                for variant in (False, "fma"):
                    plan2 = plan_cls(model, eng, dtype=dtype, use_stem=variant)
                    assert plan2.stem_mma is None
                    eng.planes.copy_(x32.to(dtype))
                    plan2(eng)
                    check("plan bf16, stem %s" % variant, dtype)
        if blocks <= 4:
            # the un-fused evaluator (plain module on the same planes) must agree too
            ev = DeviceEvaluator(model, eng, dtype=dtype, channels_last=True)
            eng.planes.copy_(x32.to(dtype))
            ev(eng)
            check("module " + dn, dtype)
    eng.close()


@pytest.mark.parametrize("board,cout,dtype", [((3, 3), 256, "bf16"), ((5, 5), 64, "bf16"), ((2, 3), 128, "fp16"), ((4, 6), 512, "bf16")])
def test_stem_mma_kernel_matches_conv(board, cout, dtype):
    """dbaz_nn_stem_mma (leaf gather + conv0 + folded affines + ReLU as one tensor-core implicit GEMM from packed states)
    against F.conv2d in fp32 on the feature planes of the same states, with the weights rounded to the storage dtype as
    the kernel sees them.  Tolerance: fp32 accumulation order + one output rounding (2^-8 relative for bf16)."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import torch.nn.functional as F
    from dotsboxesaz_b200 import engine
    from dotsboxesaz_b200.nn import _stem_mma_table
    dt = torch.bfloat16 if dtype == "bf16" else torch.float16
    n = 777  # not a multiple of the 16-row tile
    eng = engine.Engine(board, n_games=4, max_nodes=8)
    g = torch.Generator(device="cuda").manual_seed(5)
    st = eng.new_states(n)
    for ply in range(9):
        legal = eng.valid_moves(st).float()
        mv = torch.multinomial(legal + 1e-9, 1, generator=g).reshape(-1).int()
        eng.play(st, torch.where((torch.arange(n, device="cuda") % 10 > ply) & (legal.sum(1) > 0), mv, torch.full_like(mv, -1)))
    conv = torch.nn.Conv2d(3, cout, 3, padding=1).cuda()
    s_in, t_in = torch.rand(3, device="cuda", generator=g) + 0.5, torch.randn(3, device="cuda", generator=g) * 0.3
    s_o, t_o = torch.rand(cout, device="cuda", generator=g) + 0.5, torch.randn(cout, device="cuda", generator=g) * 0.2
    tab = _stem_mma_table(conv, s_in, t_in, s_o, t_o).to(dt)
    out = torch.empty((n, eng.rows, eng.cols, cout), dtype=dt, device="cuda")
    eng.nn_stem_mma(st, eng.nn_stem_mma_pack(tab), out)
    # reference from the ROUNDED table: un-fold it into a conv over [plane0, plane1, plane2, in-board indicator]
    t32 = tab.float()
    w = torch.zeros((cout, 4, 3, 3), device="cuda")
    w[:, :2] = t32[0:18].reshape(2, 3, 3, cout).permute(3, 0, 1, 2)
    w[:, 2] = t32[18:27].reshape(3, 3, cout).permute(2, 0, 1)
    w[:, 3] = t32[27:36].reshape(3, 3, cout).permute(2, 0, 1)
    x = eng.features(st, torch.float32)
    x4 = torch.cat([x, torch.ones_like(x[:, :1])], 1)
    ref = F.relu(F.conv2d(x4, w, t32[36], padding=1)).permute(0, 2, 3, 1)
    err = (out.float() - ref).abs()
    assert (err <= 2 ** -7 * (1 + ref.abs())).all(), err.max().item()
    # and the fold itself: relu(s_o * (conv(s_in * x + t_in) + b) + t_o) in fp32, up to the rounding of the table
    with torch.no_grad():
        full = F.relu(s_o.view(1, -1, 1, 1) * conv(x * s_in.view(1, 3, 1, 1) + t_in.view(1, 3, 1, 1)) + t_o.view(1, -1, 1, 1))
    assert (out.float() - full.permute(0, 2, 3, 1)).abs().max().item() < 0.25
    eng.close()


# ---------------------------------------------------------------- heads kernels against float64
# Boards by number of actions A: 8, 32, 72 (3 actions per lane), 96 (exactly 3 full lanes), 98 and 128 (the fourth slot).
HEADS_BOARDS = [(1, 1), (3, 3), (5, 5), (5, 7), (6, 6), (7, 7)]
HEADS_DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}
# Prior bound from the documented error of __expf (2 + floor(1.16 |x|) ulp, |x| <= 90 here), the fp32 rounding of x - max,
# the warp sum and the reciprocal, with an absolute floor where the kernel's exponential flushes to zero (p < 2^-126).  The
# other three are about 4x the largest error measured on a B200 (profiles/r02_net_errors.md, all 18 boards x dtypes):
# sum of priors 2.6e-7, tanh value 1.0e-7 (tanhf: 2 ulp documented), value MLP 7.1e-7 of sum |relu(h_j) w_j|.
PRIOR_REL, PRIOR_ABS = 1e-5, 1e-37
PRIOR_SUM = 1e-6
TANH_ABS = 4e-7
MLP_REL = 3e-6


def _logit_rows(n, A, cols, g, offset=0):
    """[n, cols] float64: row i takes pattern (i + offset) % 4 in its first A columns -- all equal, scale 1, one dominant
    action (+30), a spread from 0 down to -90 (where the exponential underflows) -- and a value pre-activation in the rest."""
    x = torch.randn((n, cols), dtype=torch.float64, generator=g)
    pat = (torch.arange(n) + offset) % 4
    eq = pat == 0
    x[eq, :A] = torch.randn((int(eq.sum()), 1), dtype=torch.float64, generator=g) * 3
    dom = pat == 2
    hot = torch.randint(0, A, (int(dom.sum()),), generator=g)
    x[dom.nonzero().reshape(-1), hot] = 30.0
    spread = (pat == 3).nonzero().reshape(-1)
    for i in spread.tolist():
        x[i, :A] = -90.0 * torch.rand(A, dtype=torch.float64, generator=g)
        x[i, int(torch.randint(0, A, (1,), generator=g))] = 0.0
    return x, pat


def _heads_case(eng, n, ld, dtype, g, offset, mlp=None):
    """Run nn_heads (mlp None) or nn_heads_mlp (mlp = (n_hidden, v_w)) on [n, ld] logits with NaN past the used columns;
    return the kernel's outputs (sentinel rows checked) and the float64 reference of the logits as the kernel reads them."""
    A = eng.A
    used = A + (1 if mlp is None else mlp[0])
    x, pat = _logit_rows(n, A, used, g, offset)
    full = torch.full((n, ld), float("nan"), dtype=torch.float64)
    full[:, :used] = x
    logits = full.to(dtype).cuda()
    xr = full[:, :used].to(dtype).double()  # what the kernel reads
    priors = torch.full((n + 3, A), -7.0, dtype=torch.float32, device="cuda")
    values = torch.full((n + 3,), -7.0, dtype=torch.float32, device="cuda")
    if mlp is None:
        eng.nn_heads(logits, priors, values)
    else:
        eng.nn_heads_mlp(logits, mlp[0], mlp[1], priors, values)
    torch.cuda.synchronize()
    p, v = priors.double().cpu(), values.double().cpu()
    assert (p[n:] == -7.0).all() and (v[n:] == -7.0).all(), "the kernel wrote past row n"
    p_ref = torch.softmax(xr[:, :A], dim=1)
    if mlp is None:
        return p[:n], v[:n], p_ref, torch.tanh(xr[:, A]), None, pat
    w = mlp[1].double().cpu()
    terms = torch.relu(xr[:, A:]) * w[:-1]
    return p[:n], v[:n], p_ref, torch.tanh(terms.sum(1) + w[-1]), terms.abs().sum(1), pat


@pytest.mark.parametrize("dtype", list(HEADS_DTYPES))
@pytest.mark.parametrize("board", HEADS_BOARDS)
def test_heads_kernels_match_float64(board, dtype):
    """k_nn_heads and k_nn_heads_mlp against the float64 softmax / tanh / value MLP of the logits rounded to the input
    dtype: ld = A + (1 or n_hidden), that rounded up to 8, and a larger odd ld with NaN in the unused columns; 1, 7 and 8193
    rows (not a multiple of the 8 rows of a block); every logit pattern; n_hidden 1, 8, 31, 32.  Nothing is written past
    row n.  All-equal logits give a uniform row."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine
    dt = HEADS_DTYPES[dtype]
    eng = engine.Engine(board, n_games=1, max_nodes=4)
    A = eng.A
    assert A == 2 * (board[0] + 1) * (board[1] + 1)
    g = torch.Generator().manual_seed(A * 7 + len(dtype))
    worst = {"prior_rel": 0.0, "prior_sum": 0.0, "tanh": 0.0, "mlp_rel": 0.0}
    try:
        for n_hidden in (None, 1, 8, 31, 32):
            used = A + (1 if n_hidden is None else n_hidden)
            mlp = None
            if n_hidden is not None:
                v_w = (torch.randn(n_hidden + 1, generator=g) * 0.5).float().cuda()
                mlp = (n_hidden, v_w)
            for ld in sorted({used, (used + 7) // 8 * 8, used + 14 + (used + 1) % 2}):
                for n in (1, 7, 8193):
                    for offset in (range(4) if n < 8 else (0,)):
                        p, v, p_ref, v_ref, v_scale, pat = _heads_case(eng, n, ld, dt, g, offset, mlp)
                        where = (board, dtype, n_hidden, ld, n, offset)
                        assert torch.isfinite(p).all() and torch.isfinite(v).all(), where
                        err = (p - p_ref).abs()
                        bad = (err > PRIOR_REL * p_ref + PRIOR_ABS).nonzero()
                        assert bad.numel() == 0, (where, "prior", bad[0].tolist(), p[tuple(bad[0])].item(), p_ref[tuple(bad[0])].item())
                        eq = p[pat == 0]
                        assert (eq == eq[:, :1]).all(), (where, "all-equal logits give a non-uniform row")
                        s = (p.sum(1) - 1).abs().max().item()
                        assert s <= PRIOR_SUM, (where, "sum", s)
                        verr = (v - v_ref).abs()
                        if v_scale is None:
                            assert (verr <= TANH_ABS).all(), (where, "tanh value", verr.max().item())
                            worst["tanh"] = max(worst["tanh"], verr.max().item())
                        else:
                            assert (verr <= MLP_REL * v_scale + TANH_ABS).all(), (where, "MLP value", verr.max().item())
                            sel = v_scale > 0.1
                            if sel.any():
                                worst["mlp_rel"] = max(worst["mlp_rel"], (verr[sel] / v_scale[sel]).max().item())
                        big = p_ref > 1e-30
                        worst["prior_rel"] = max(worst["prior_rel"], (err[big] / p_ref[big]).max().item())
                        worst["prior_sum"] = max(worst["prior_sum"], s)
        _record("heads A=%d %s" % (A, dtype), worst)
    finally:
        eng.close()


def test_heads_rejects_logits_without_value_column():
    """[n, A] logits have no column A for the value pre-activation: nn_heads must refuse them instead of reading the next
    row's first logit as the value."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dotsboxesaz_b200 import engine
    eng = engine.Engine((7, 7), n_games=4, max_nodes=8)
    try:
        logits = torch.zeros((4, eng.A), dtype=torch.float32, device="cuda")
        with pytest.raises(engine.EngineError, match="ld >= A \\+ 1"):
            eng.nn_heads(logits, torch.empty((4, eng.A), device="cuda"), torch.empty((4,), device="cuda"))
        eng.nn_heads(torch.zeros((4, eng.A + 1), device="cuda"), torch.empty((4, eng.A), device="cuda"), torch.empty((4,), device="cuda"))
        with pytest.raises(engine.EngineError):
            eng.nn_heads_mlp(logits, 8, torch.zeros(9, device="cuda"), torch.empty((4, eng.A), device="cuda"), torch.empty((4,), device="cuda"))
    finally:
        eng.close()
