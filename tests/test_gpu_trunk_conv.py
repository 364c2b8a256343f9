"""The trunk convolution kernel (dbaz_nn_trunk_conv: a tcgen05 GEMM per output position over its in-board taps) against a
float64 reference on bf16-rounded weights and inputs (nn.trunk_conv_reference), its row independence, the rows it must not
write, and FusedSimpleNN with and without it."""
import pytest
import torch

pytestmark = pytest.mark.gpu

NS = [1, 127, 128, 255, 256, 257, 1000, 4096]
SENTINEL = -12352.0  # exactly representable in bf16


def _layer(eng, hi, wi, pad, cap, seed):
    from dotsboxesaz_b200.nn import trunk_conv_pack
    dev = eng.device
    ho, wo = hi + 2 * pad - 2, wi + 2 * pad - 2
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.rand(cap, hi, wi, 256, generator=g).to(torch.bfloat16).to(dev)
    w = (torch.randn(256, 256, 3, 3, generator=g) * 0.03).to(dev)
    bias = ((torch.randn(ho * wo, 256, generator=g) * 0.3).to(dev), (torch.randn(256, generator=g) * 0.3).to(dev))
    y = torch.full((cap, ho, wo, 256), SENTINEL, dtype=torch.bfloat16, device=dev)
    wp = trunk_conv_pack(w)
    plan = eng.nn_trunk_conv_plan(x, y, wp, bias[0], bias[1], pad)
    return x, w, bias, y, plan


@pytest.fixture(scope="module")
def eng():
    from dotsboxesaz_b200 import engine
    e = engine.Engine((3, 3), n_games=8, max_nodes=16)
    yield e
    e.close()


@pytest.mark.parametrize("board", [(3, 3), (5, 5), (2, 3), (7, 7)])
@pytest.mark.parametrize("pad", [1, 0])
def test_layer_matches_reference(eng, board, pad):
    """Every n: at most one bf16 rounding step from the reference, and rows n .. cap-1 keep the sentinel."""
    from dotsboxesaz_b200.nn import trunk_conv_reference
    hi, wi = board[0] + 1, board[1] + 1
    cap = 4096 + 37
    x, w, bias, y, plan = _layer(eng, hi, wi, pad, cap, seed=hi * 10 + wi + pad)
    ref = trunk_conv_reference(x[:4096], w, *bias, pad).float()
    for n in NS:
        y.fill_(SENTINEL)
        out = eng.nn_trunk_conv(plan, n)
        torch.cuda.synchronize()
        assert eng.status()["errors"] == 0
        r = ref[:n]
        err = (out.float() - r).abs()
        # one bf16 rounding step of each value (8 significant bits), measured against the value's own magnitude
        bound = torch.clamp(r.abs(), min=2.0 ** -10) * 2.0 ** -7
        assert bool((err <= bound).all()), (board, pad, n, err.max().item(), (err - bound).max().item())
        assert bool((y[n:].float() == SENTINEL).all()), (board, pad, n)


def test_rows_are_independent_and_launches_repeat(eng):
    """Copies of the same boards at scattered rows and in batches of different n give bit-identical outputs."""
    hi = wi = 4
    cap = 3000
    x, w, bias, y, plan = _layer(eng, hi, wi, 1, cap, seed=7)
    base = x[:64].clone()
    n0 = 64
    out0 = eng.nn_trunk_conv(plan, n0).clone()
    again = eng.nn_trunk_conv(plan, n0).clone()
    assert torch.equal(out0.view(torch.int16), again.view(torch.int16))
    g = torch.Generator(device="cpu").manual_seed(11)
    for n in (300, 1111, 2999):
        rows = torch.randperm(n, generator=g)[:64].to(eng.device)
        x[rows] = base
        out = eng.nn_trunk_conv(plan, n)
        assert torch.equal(out[rows].view(torch.int16), out0.view(torch.int16)), n
    x2, _, _, _, _ = _layer(eng, hi, wi, 1, cap, seed=7)  # fresh inputs again: rows 0..63 are the original boards
    x.copy_(x2)
    assert torch.equal(eng.nn_trunk_conv(plan, cap)[:64].view(torch.int16), out0.view(torch.int16))


def test_plan_rejects_bad_buffers(eng):
    from dotsboxesaz_b200.engine import EngineError
    x, w, bias, y, plan = _layer(eng, 4, 4, 1, 256, seed=1)
    with pytest.raises(ValueError):
        eng.nn_trunk_conv_plan(x, y[:, :2], w, *bias, 1)
    with pytest.raises(ValueError):
        eng.nn_trunk_conv_plan(x.float(), y, w, *bias, 1)
    with pytest.raises(ValueError):
        eng.nn_trunk_conv_plan(x, y, w, bias[0], bias[1][:128], 1)
    with pytest.raises(EngineError):
        eng.nn_trunk_conv(plan, 257)


@pytest.mark.parametrize("board", [(3, 3), (5, 5)])
def test_fused_simple_nn_uses_the_kernel_and_reloads(board):
    """The bf16 plan runs the trunk kernel for conv1-conv3 at TRUNK_MIN_ROWS leaves; it agrees with the cuDNN plan, and
    load() of new weights gives bit for bit what a fresh plan gives."""
    from dotsboxesaz_b200 import engine
    from dotsboxesaz_b200.dots_boxes.dots_boxes_nn import SimpleNN
    from dotsboxesaz_b200.nn import FusedSimpleNN
    torch.manual_seed(3)
    n = FusedSimpleNN.TRUNK_MIN_ROWS + 256
    eng = engine.Engine(board, n_games=n, max_nodes=64)
    try:
        model = SimpleNN(board=board)
        with torch.no_grad():
            for m in model.modules():
                if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
                    m.running_mean.uniform_(-0.5, 0.5); m.running_var.uniform_(0.5, 2.0)
                    m.weight.uniform_(0.5, 1.5); m.bias.uniform_(-0.2, 0.2)
        model.eval()
        states = eng.new_states(n)
        rng = torch.Generator().manual_seed(1)
        moves = torch.full((n,), -1, dtype=torch.int32)
        valid = eng.valid_moves(states).cpu()
        for g in range(n):
            choices = valid[g].nonzero().flatten()
            if g % 3 and len(choices):
                moves[g] = int(choices[torch.randint(len(choices), (1,), generator=rng)])
        eng.play(states, moves.numpy())
        eng.leaf_states[:n] = states
        eng._batch_rows = n

        def run(ev):
            ev(eng)
            torch.cuda.synchronize()
            return eng.priors[:n].clone(), eng.values[:n].clone()

        ev = FusedSimpleNN(model, eng)
        assert len(ev.trunk) == 3 and ev.engine_launches == 5
        lib = FusedSimpleNN(model, eng, use_trunk=False)
        assert lib.trunk is None
        (p1, v1), (p0, v0) = run(ev), run(lib)
        # same bf16-rounded biases and the accumulation order of cuDNN's default implicit GEMM for these convs: the same
        # numbers when cuDNN runs that algorithm (as bench.py's runs do); another algorithm cuDNN may choose under other
        # global settings sums in another order, so allow a few bf16 rounding flips
        dp, dv = (p1 - p0).abs().max().item(), (v1 - v0).abs().max().item()
        print("plan vs library: max |dp| %.3g, max |dv| %.3g, equal %s" % (dp, dv, torch.equal(p1, p0) and torch.equal(v1, v0)))
        assert dp < 0.02 and dv < 0.05, (dp, dv)
        with torch.no_grad():
            for prm in model.parameters():
                prm.mul_(0.9)
        ev.load(model)
        pr, vr = run(ev)
        pf, vf = run(FusedSimpleNN(model, eng))
        assert torch.equal(pr, pf) and torch.equal(vr, vf)
        assert eng.status()["errors"] == 0
    finally:
        eng._batch_rows = None
        eng.close()


def test_layer_beyond_one_chunk(eng):
    """Past 4096 boards the items run in chunks of 4096 boards: every chunk, the partial last one too, matches the reference
    and leaves the rows past n alone."""
    from dotsboxesaz_b200.nn import trunk_conv_reference
    cap = 9000
    x, w, bias, y, plan = _layer(eng, 4, 4, 1, cap, seed=21)
    ref = trunk_conv_reference(x, w, *bias, 1).float()
    for n in (4097, 8191, 8999):
        y.fill_(SENTINEL)
        out = eng.nn_trunk_conv(plan, n).float()
        torch.cuda.synchronize()
        err = (out - ref[:n]).abs()
        bound = torch.clamp(ref[:n].abs(), min=2.0 ** -10) * 2.0 ** -7
        assert bool((err <= bound).all()), (n, err.max().item())
        assert bool((y[n:].float() == SENTINEL).all()), n
