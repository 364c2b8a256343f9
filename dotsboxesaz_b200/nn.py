"""Policy/value nets and the inference wrapper (reference: nn.py, dots_boxes/dots_boxes_nn.py).

The nets are the only dense contraction of the path and stay plain PyTorch (cuDNN / cuBLAS
on the tensor cores); module and parameter names equal the reference's so that its
`model_gen{g}.pt` checkpoints (`{'last_batch_idx', 'model_dict', 'optimizer_dict'}`,
nn.py:293-295) load unchanged.  `DeviceEvaluator` is the engine-facing replacement of
AsyncBatchedProxy + NeuralNetWrapper.predict_sync (utils/proxies.py:34-72, nn.py:155-160):
it reads the leaf planes the select kernel wrote, runs the net in eval mode, and writes
exp(log p) and v into the engine's float32 buffers -- all on the current stream, with no
host round trip, so Engine.run_search can capture whole waves in a CUDA graph.
"""
import asyncio
import copy
import logging
import os

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

logger = logging.getLogger(__name__)


def _conv(in_ch, out_ch, k, groups=1, padding=True):
    # nn.py:61-71: odd kernels use symmetric padding, even kernels pad right/bottom
    if k % 2 == 1:
        return nn.Conv2d(in_ch, out_ch, k, padding=(k - 1) // 2 if padding else 0, groups=groups)
    conv = nn.Conv2d(in_ch, out_ch, k, padding=0, groups=groups)
    if not padding:
        return conv
    return nn.Sequential(nn.ConstantPad2d((0, k // 2, 0, k // 2), 0.0), conv)


class ResBlock(nn.Module):
    """nn.py:33-58"""

    def __init__(self, nb_channels, kernel_size, n_groups, inner_channels):
        super().__init__()
        inner = inner_channels if inner_channels else nb_channels
        self.inner_conv = None
        if inner_channels:
            self.inner_conv = _conv(inner, inner, kernel_size, n_groups)
            self.inner_bn = nn.BatchNorm2d(inner)
        self.conv1 = _conv(nb_channels, inner, kernel_size, n_groups)
        self.bn1 = nn.BatchNorm2d(inner)
        self.conv2 = _conv(inner, nb_channels, kernel_size, n_groups)
        self.bn2 = nn.BatchNorm2d(nb_channels)

    def forward(self, x):
        y = F.relu(self.bn1(self.conv1(x)))
        if self.inner_conv is not None:
            y = F.relu(self.inner_bn(self.inner_conv(y)))
        y = self.bn2(self.conv2(y))
        return F.relu(y + x)


class ResNet(nn.Module):
    """nn.py:16-30"""

    def __init__(self, in_channels, nb_channels, kernel_size, nb_blocks, n_groups=1, inner_channels=None, pad_layer0=True):
        super().__init__()
        self.conv0 = _conv(in_channels, nb_channels, 3, 1, pad_layer0)
        self.bn0 = nn.BatchNorm2d(nb_channels)
        self.resblocks = nn.Sequential(*(ResBlock(nb_channels, kernel_size, n_groups, inner_channels) for _ in range(nb_blocks)))

    def forward(self, x):
        return self.resblocks(F.relu(self.bn0(self.conv0(x))))


class PolicyHead(nn.Module):
    """nn.py:74-87"""

    def __init__(self, in_channels, inner_channels, fc_in, nb_actions):
        super().__init__()
        self.conv0 = nn.Conv2d(in_channels, inner_channels, kernel_size=(1, 1))
        self.bn0 = nn.BatchNorm2d(inner_channels)
        self.fc = nn.Linear(fc_in, nb_actions)

    def forward(self, x):
        x = F.relu(self.bn0(self.conv0(x)))
        return F.log_softmax(self.fc(x.reshape(x.size(0), -1)), dim=1)


class ValueHead(nn.Module):
    """nn.py:90-105"""

    def __init__(self, in_channels, inner_channels, fc_in, fc_inner):
        super().__init__()
        self.conv0 = nn.Conv2d(in_channels, inner_channels, kernel_size=(1, 1))
        self.bn0 = nn.BatchNorm2d(inner_channels)
        self.fc0 = nn.Linear(fc_in, fc_inner)
        self.fc1 = nn.Linear(fc_inner, 1)

    def forward(self, x):
        x = F.relu(self.bn0(self.conv0(x)))
        x = F.relu(self.fc0(x.reshape(x.size(0), -1)))
        return torch.tanh(self.fc1(x))


def _load_parameters(model, generation, to_device=None):
    fn = model.params.nn.chkpts_filename.format(generation)
    logger.info("Model loaded from: %s", fn)
    model.load_state_dict(torch.load(fn, map_location="cpu")["model_dict"])
    model.to(to_device)


class ResNetZero(nn.Module):
    """nn.py:108-129.  `params.nn.model_parameters` = {resnet, value_head, policy_head} kwargs."""

    def __init__(self, params):
        super().__init__()
        self.params = params
        mp = params.nn.model_parameters
        self.bn_input = nn.BatchNorm2d(mp.resnet.in_channels)
        self.resnet = ResNet(**mp.resnet)
        self.value_head = ValueHead(**mp.value_head)
        self.policy_head = PolicyHead(**mp.policy_head)

    def forward(self, x):
        x = self.resnet(self.bn_input(x))
        return self.policy_head(x), self.value_head(x)

    def load_parameters(self, generation, to_device=None):
        _load_parameters(self, generation, to_device)


def resnet_zero_parameters(board=(3, 3), nb_channels=64, nb_blocks=20, head_channels=16, fc_inner=8):
    """model_parameters for a board of L x C boxes; (3, 3) reproduces configuration.py:133-155."""
    rows, cols = board[0] + 1, board[1] + 1
    fc_in = head_channels * rows * cols
    return {"resnet": {"pad_layer0": True, "in_channels": 3, "nb_channels": nb_channels, "inner_channels": None,
                       "kernel_size": 3, "nb_blocks": nb_blocks, "n_groups": 1},
            "policy_head": {"in_channels": nb_channels, "inner_channels": head_channels, "fc_in": fc_in,
                            "nb_actions": 2 * rows * cols},
            "value_head": {"in_channels": nb_channels, "inner_channels": head_channels, "fc_in": fc_in, "fc_inner": fc_inner}}


class AlphaZeroLoss(nn.Module):
    """nn.py:131-138"""

    def forward(self, p, v, pi, z):
        loss_v = (z - v).pow(2).mean()
        loss_pi = -(pi * p).sum(1).mean()
        return loss_v + loss_pi, (loss_pi.item(), loss_v.item())


class _NullWriter:
    def add_scalar(self, *a, **k):
        pass

    def add_scalars(self, *a, **k):
        pass

    def add_text(self, *a, **k):
        pass


class NeuralNetWrapper:
    """nn.py:145-274: host-facing predict API (numpy in, numpy out) and the supervised training step of a
    generation (SGD, AlphaZeroLoss, one random board symmetry per batch, checkpoint per generation).  Plain
    PyTorch: training is not on the self-play hot path."""

    def __init__(self, model, params):
        self.params = params
        self.device = torch.device(params.nn.pytorch_device if torch.cuda.is_available() else "cpu")
        self.model = model.to(self.device) if model is not None else None

    def set_model(self, model):
        self.model = model.to(self.device)

    @torch.no_grad()
    def predict_sync(self, X):
        self.model.train(False)
        x = torch.as_tensor(np.asarray(X), dtype=torch.float32, device=self.device)
        p, v = self.model(x)
        return torch.exp(p).cpu().numpy(), v.cpu().numpy()

    async def predict(self, X):
        return await asyncio.get_event_loop().run_in_executor(None, self.predict_sync, X)

    async def predict_from_game(self, game_state):
        return await self.predict([game_state.get_features()])

    async def __call__(self, X):
        return await self.predict(X)

    def train(self, train_dataset, val_dataset, writer, generation):
        """nn.py:175-274.  Returns the running batch index (stored in the checkpoint)."""
        import torch.utils.data as data
        writer = writer or _NullWriter()
        tp = self.params.nn.train_params
        # datasets that live on the device (samples.DeviceDataset) hand out shuffled device batches themselves; anything
        # else goes through a DataLoader as in the reference (nn.py:177-181)
        class _Batches:
            def __init__(self, ds, bs, shuffle):
                self.ds, self.bs, self.shuffle = ds, bs, shuffle

            def __iter__(self):
                return self.ds.batches(self.bs, shuffle=self.shuffle, drop_last=True)

        def loader(ds, bs, shuffle):
            if hasattr(ds, "batches"):
                return _Batches(ds, bs, shuffle)
            return data.DataLoader(ds, bs, shuffle=shuffle, drop_last=True)
        train_data = loader(train_dataset, tp.train_batch_size, True)
        val_data = loader(val_dataset, tp.val_batch_size, False) if val_dataset is not None else None
        criterion = AlphaZeroLoss()
        optimizer = torch.optim.SGD(self.model.parameters(), lr=tp.lr, **tp.optimizer_params)
        batch_i = 0
        if generation > 0:
            batch_i = load_checkpoint(self.params.nn.chkpts_filename.format(generation - 1), self.model, optimizer, self.device)
        writer.add_scalar("lr", tp.lr, batch_i)

        def accuracy(v, z, threshold=0.5):
            ok = z.sign().eq(v.sign()) & (v - z).abs().lt(threshold)
            return ok.sum().item(), z.size(0)

        for epoch in range(min(2 * generation, tp.nb_epochs)):
            self.model.train(True)
            tr_loss, tr_batches, tr_ok, tr_tot = 0.0, 0, 0, 1
            for boards, pi, z in train_data:
                batch_i += 1
                tr_batches += 1
                boards, pi, z = boards.to(self.device), pi.to(self.device), z.to(self.device)
                boards, pi = tp.symmetries(boards, pi)
                p, v = self.model(boards)
                loss, (loss_pi, loss_v) = criterion(p, v, pi, z)
                loss.backward()
                optimizer.step()
                optimizer.zero_grad()
                with torch.no_grad():
                    c, t = accuracy(v, z)
                tr_ok += c; tr_tot += t
                tr_loss += loss_pi + loss_v
                writer.add_scalars("loss", {"pi/train": loss_pi, "v/train": loss_v, "total/train": loss_pi + loss_v}, batch_i)
            val_loss, va_ok, va_tot = 0.0, 0, 1
            if val_data is not None:
                self.model.train(False)
                lv = lp = 0.0
                nb = 0
                with torch.no_grad():
                    for boards, pi, z in val_data:
                        nb += 1
                        boards, pi, z = boards.to(self.device), pi.to(self.device), z.to(self.device)
                        boards, pi = tp.symmetries(boards, pi)
                        p, v = self.model(boards)
                        c, t = accuracy(v, z)
                        va_ok += c; va_tot += t
                        _, (a, b) = criterion(p, v, pi, z)
                        lp += a; lv += b
                if nb:
                    val_loss = (lp + lv) / nb
                    writer.add_scalars("loss", {"pi/eval": lp / nb, "v/eval": lv / nb, "total/eval": val_loss}, batch_i)
            writer.add_scalars("accuracy", {"v/train": tr_ok / tr_tot, "v/eval": va_ok / va_tot}, batch_i)
            writer.add_scalar("generation", generation, batch_i)
            print(f"Epoch {epoch}, train loss= {tr_loss / max(tr_batches, 1):5f}, validation loss= {val_loss:5f}", flush=True)
        save_checkpoint(self.params.nn.chkpts_filename.format(generation), self.model, optimizer, batch_i)
        return batch_i


class GenerationLrScheduler:
    """nn.py:276-290"""

    def __init__(self, schedule):
        assert schedule is not None
        self.schedule = schedule

    def __call__(self, generation):
        lr = None
        for g in range(generation + 1):
            lr = self.schedule.get(g, lr)
        assert lr is not None
        return lr

    def __repr__(self):
        return f"GenerationLrScheduler({self.schedule})"


def save_checkpoint(filename, model, optimizer, last_batch_idx):
    torch.save({"last_batch_idx": last_batch_idx, "model_dict": model.state_dict(), "optimizer_dict": optimizer.state_dict()},
               filename)


def load_checkpoint(filename, model, optimizer, to_device):
    if not os.path.isfile(filename):
        raise ValueError(f"=> no checkpoint found at '{filename}'")
    ck = torch.load(filename, map_location="cpu")
    model.load_state_dict(ck["model_dict"])
    optimizer.load_state_dict(ck["optimizer_dict"])
    model.to(to_device)
    for state in optimizer.state.values():
        for k, v in state.items():
            if isinstance(v, torch.Tensor):
                state[k] = v.to(to_device)
    return ck["last_batch_idx"]


# ----------------------------------------------------------------- engine side
class DeviceEvaluator:
    """Leaf evaluation for the lock-step search: engine.planes -> net -> engine.priors / engine.values.

    dtype: compute dtype of the net (torch.bfloat16 default; float32 reproduces the reference's
    arithmetic type).  The select kernel writes the planes directly in this dtype and, with
    channels_last, directly in NHWC, so no cast / permute kernels run before the first conv.
    """

    def __init__(self, model, engine, dtype=torch.bfloat16, channels_last=True):
        self.engine = engine
        self.dtype = dtype
        self.model = copy.deepcopy(model).to(engine.device).train(False)  # never move, retype or freeze the caller's (training) module
        if dtype != torch.float32:
            self.model = self.model.to(dtype)
        if channels_last:
            self.model = self.model.to(memory_format=torch.channels_last)
        for p in self.model.parameters():
            p.requires_grad_(False)
        engine.set_planes(dtype, channels_last)

    @torch.no_grad()
    def __call__(self, eng):
        """Capturable: fixed input/output addresses, no host sync (Engine.run_search(graph_waves=...))."""
        logp, v = self.model(eng.planes)
        torch.exp(logp.float(), out=eng.priors)  # nn.py:159: probabilities, float32
        eng.values.copy_(v.reshape(-1))


def _bn_affine(bn):
    """Eval-mode BatchNorm as y = scale*x + shift (float32)."""
    scale = (bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps))
    shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
    return scale.contiguous(), shift.contiguous()


def _stem_tables(conv, rows, cols, in_scale=None, in_shift=None):
    """Host-side folding for Engine.nn_stem (float32, exact algebra): the conv over the three input planes
    becomes  y[p] = B[p] + k*K2[p] + sum over set edge bits of W01[c][tap]  -- see dbaz_nn_kernels.cuh."""
    w = conv.weight.detach().float()                       # [cout, 3, 3, 3]
    dev = w.device
    s = torch.ones(3, device=dev) if in_scale is None else in_scale.float()
    t = torch.zeros(3, device=dev) if in_shift is None else in_shift.float()
    ws = w * s.view(1, 3, 1, 1)
    pad = conv.padding
    e2 = torch.zeros((1, 3, rows, cols), device=dev); e2[0, 2] = 1.0
    k2 = F.conv2d(e2, ws, None, padding=pad)[0]            # [cout, H, W]: plane-2 weights summed over in-board taps
    tmap = t.view(1, 3, 1, 1).expand(1, 3, rows, cols).contiguous()
    b = conv.bias.detach().float().view(-1, 1, 1) + F.conv2d(tmap, w, None, padding=pad)[0]
    w01 = ws[:, :2].permute(1, 2, 3, 0).reshape(18, -1).contiguous()          # [c][ky][kx][cout]
    to_pos = lambda x: x.permute(1, 2, 0).reshape(rows * cols, -1).contiguous()  # [H*W][cout]
    return w01, to_pos(b), to_pos(k2)


_ONE = (1, 1)


def _conv_relu(x, w, b, pad):
    """relu(conv(x, w) + b) as ONE library kernel (cuDNN's fused conv-bias-activation; same speed as the bare conv)."""
    return torch.cudnn_convolution_relu(x, w, b, _ONE, pad, _ONE, 1)


def _conv_add_relu(x, w, z, b, pad):
    """relu(conv(x, w) + z + b) as ONE library kernel (z has the shape of the output)."""
    return torch.cudnn_convolution_add_relu(x, w, z, 1.0, b, _ONE, pad, _ONE, 1)


def _cl(w, dtype):
    return w.to(dtype).contiguous(memory_format=torch.channels_last)


def _stem_mma_table(conv, in_scale=None, in_shift=None, out_scale=None, out_shift=None):
    """Folded weights [48, cout] (float32) of Engine.nn_stem_mma for  relu(out_scale * (conv(in_scale * x + in_shift) + b) +
    out_shift)  with zero padding applied AFTER the input affine (nn.py:118-119): rows 0-17 edge-plane taps, 18-26 third-plane
    taps, 27-35 per-tap constants for in-board taps (image of in_shift), 36 bias.  See dbaz_nn_kernels.cuh."""
    w = conv.weight.detach().float()                       # [cout, 3, 3, 3]
    dev, cout = w.device, w.shape[0]
    s = torch.ones(3, device=dev) if in_scale is None else in_scale.float()
    t = torch.zeros(3, device=dev) if in_shift is None else in_shift.float()
    so = torch.ones(cout, device=dev) if out_scale is None else out_scale.float()
    to = torch.zeros(cout, device=dev) if out_shift is None else out_shift.float()
    ws = w * s.view(1, 3, 1, 1)
    tab = torch.zeros((48, cout), device=dev)
    tab[0:18] = ws[:, :2].permute(1, 2, 3, 0).reshape(18, cout)           # [plane][ky][kx]
    tab[18:27] = ws[:, 2].permute(1, 2, 0).reshape(9, cout)
    tab[27:36] = (w * t.view(1, 3, 1, 1)).sum(1).permute(1, 2, 0).reshape(9, cout)
    tab[36] = conv.bias.detach().float()
    tab = tab * so.view(1, cout)
    tab[36] += to
    return tab.contiguous()


def _stem_mma_ok(conv, engine, dtype):
    return (dtype in (torch.bfloat16, torch.float16) and not isinstance(conv, nn.Sequential) and tuple(conv.padding) == (1, 1)
            and conv.kernel_size == (3, 3) and conv.in_channels == 3 and conv.out_channels % 64 == 0 and conv.out_channels <= 512)


def tower_pack(w3, b3, w_head=None, b_head=None):
    """Weights of the fused residual-tower kernel in the order include/dbaz_b200.h (dbaz_nn_tower) documents.
    w3 float32 [S, 64, 64, 3, 3], b3 float32 [S, 64]: the S conv stages with their BatchNorm folded in;
    w_head [hc, 64], b_head [hc]: the 1x1 head convolution (optional).  Returns (packed uint8 [bytes], bias float32 [S(+1), 64])."""
    S = w3.shape[0]
    assert tuple(w3.shape[1:]) == (64, 64, 3, 3)
    x = w3.reshape(S, 64, 4, 2, 8, 3, 3).permute(0, 6, 2, 3, 5, 1, 4)      # [S, kx, ks, kh, ky, co, i]
    x = torch.flip(x, dims=(4,)).reshape(S, 12, 2, 192, 8)                  # rows: ky = 2, 1, 0
    parts = [x.to(torch.bfloat16).contiguous().view(torch.uint8).reshape(-1)]
    bias = [b3.float()]
    if w_head is not None:
        hc = w_head.shape[0]
        h = w_head.reshape(hc, 4, 2, 8).permute(1, 2, 0, 3)                 # [ks, kh, co, i]
        parts.append(h.to(torch.bfloat16).contiguous().view(torch.uint8).reshape(-1))
        bh = torch.zeros((1, 64), dtype=torch.float32, device=b3.device)
        bh[0, :hc] = b_head.float()
        bias.append(bh)
    return torch.cat(parts).contiguous(), torch.cat(bias).contiguous()


def tower_reference(x_nhwc, w3, b3, w_head=None, b_head=None):
    """What the tower kernel computes, in plain PyTorch float32 on bf16-rounded weights, activations rounded to bf16
    between stages (the kernel keeps them as bf16 in shared memory).  x_nhwc [n, H, W, 64]; returns NHWC bf16."""
    r = lambda t: t.to(torch.bfloat16).float()
    x = x_nhwc.float().permute(0, 3, 1, 2)
    blk = mid = out = x
    for s in range(w3.shape[0]):
        y = F.conv2d(x if s % 2 == 0 else mid, r(w3[s]), b3[s].float(), padding=1)
        if s % 2 == 0:
            blk = x
            mid = r(F.relu(y))
            out = mid
        else:
            x = r(F.relu(y + blk))
            out = x
    if w_head is not None:
        out = r(F.relu(F.conv2d(out, r(w_head)[:, :, None, None], b_head.float())))
    return out.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def trunk_conv_pack(w):
    """[256 cout, 256 cin, 3, 3] weights -> the [ky][kx][cout][cin] bf16 order of Engine.nn_trunk_conv_plan, as [2304, 256]."""
    assert tuple(w.shape) == (256, 256, 3, 3)
    return w.permute(2, 3, 0, 1).reshape(9 * 256, 256).to(torch.bfloat16).contiguous()


def trunk_conv_bias(bias, bpos, pad):
    """The two biases of the trunk kernel as the library plan rounds them: the per-position map bpos [cout, ho, wo] (the
    image of the previous BatchNorm's shift; different at each border position of a padded layer) and the conv's bias
    [cout], each rounded to bf16 like the `z` operand and bias of cuDNN's conv-add-bias-ReLU.  pad 0: the map is one
    constant, folded into the bias as the library plan does.  Returns (bias_pos [ho * wo, cout], bias [cout]) float32."""
    r = lambda t: t.to(torch.bfloat16).float()
    cout = bpos.shape[0]
    if pad == 0:
        return torch.zeros((bpos.shape[1] * bpos.shape[2], cout), device=bpos.device), r(bias.float() + bpos[:, 0, 0].float()).contiguous()
    return r(bpos.float().permute(1, 2, 0).reshape(-1, cout)).contiguous(), r(bias.float()).contiguous()


def trunk_conv_reference(x_nhwc, w, bias_pos, bias, pad):
    """What the trunk kernel computes, in float64 on bf16-rounded weights and inputs: relu(conv(x, w) + bias_pos + bias),
    rounded once to bf16.  x_nhwc [n, hi, wi, 256]; w [256, 256, 3, 3]; bias_pos [ho * wo, 256]; bias [256]; returns
    [n, ho, wo, 256] bf16."""
    r = lambda t: t.to(torch.bfloat16).double()
    y = F.conv2d(r(x_nhwc).permute(0, 3, 1, 2), r(w), None, padding=pad)
    n, c, ho, wo = y.shape
    y = y + bias_pos.double().t().reshape(1, c, ho, wo) + bias.double().view(1, c, 1, 1)
    return F.relu(y).permute(0, 2, 3, 1).to(torch.bfloat16).contiguous()


def _copy_plan_tensors(dst, src, path="plan"):
    """dst <- src for every tensor reachable through tuples / lists / dicts of the two plans, IN PLACE (same addresses:
    CUDA graphs captured around the plan stay valid).  Structures must match; None on the src side (buffers a
    weights-only plan did not allocate) is skipped."""
    if src is None:
        return
    if isinstance(dst, torch.Tensor):
        if not isinstance(src, torch.Tensor) or dst.shape != src.shape or dst.dtype != src.dtype:
            raise RuntimeError("plan reload: %s changed shape or type" % path)
        dst.copy_(src)
    elif isinstance(dst, (tuple, list)):
        if not isinstance(src, (tuple, list)) or len(dst) != len(src):
            raise RuntimeError("plan reload: %s changed structure" % path)
        for i, (d, s_) in enumerate(zip(dst, src)):
            _copy_plan_tensors(d, s_, "%s[%d]" % (path, i))
    elif isinstance(dst, dict):
        for k in dst:
            _copy_plan_tensors(dst[k], src.get(k), "%s.%s" % (path, k))


class _ReloadablePlan:
    """load(model): fold `model`'s current weights into this plan's tensors in place.  A coach generation changes the
    weights, not the architecture, so the plan object -- and with it every CUDA graph the engine captured around it
    (keyed by the evaluator object) -- survives the update; only the folded weights are recomputed."""

    def load(self, model):
        fresh = type(self)(model, self.engine, dtype=self.dtype, _buffers=False, **self._ctor)
        for name, val in self.__dict__.items():
            if name in ("engine", "_ctor") or not isinstance(val, (torch.Tensor, tuple, list, dict)):
                continue
            _copy_plan_tensors(val, fresh.__dict__.get(name), name)
        return self


class FusedSimpleNN(_ReloadablePlan):
    """Inference plan for SimpleNN (dots_boxes_nn.py:61-98), 9 kernels per batch instead of the module's ~45.

    Every layer is conv/linear -> ReLU -> eval-mode BatchNorm (y = s*r + t).  The affine is pushed into the NEXT
    layer: its weights take the factor s per input channel and its bias takes the image of t -- a constant vector for
    the unpadded conv4 and the linear layers, a per-position map for the zero-padded 3x3 convs (the border sees fewer
    taps).  So each layer is ONE kernel on the tensor cores with its bias/ReLU in the epilogue.  In bf16 at batches of
    TRUNK_MIN_ROWS and more, the padded convs conv1-conv3 run as the engine's trunk kernel, which skips the taps that fall
    into the padding and otherwise computes what cuDNN computes (same bf16 map and bias, same order of the sums);
    otherwise they run as cuDNN's fused conv-add-bias-ReLU with the map as its `z` operand.  conv4 is cuDNN conv-bias-ReLU, the FC layers cuBLASLt GEMM-bias-ReLU; conv0 (leaf
    gather + conv + ReLU straight from the packed leaf states) and the softmax/tanh heads are the engine's own kernels.
    fc0's columns are permuted to the NHWC flatten order, policy and value heads are one GEMM.  Same function as the
    module in eval mode up to rounding of the compute dtype (tests/test_gpu_nn.py)."""

    # Below this many leaves the padded convs stay on cuDNN even when the trunk kernel is available: a work item is 128
    # boards at one position, so small batches leave most SMs idle and one 9-tap item (~16 us) is the kernel's floor.
    # tools/trunk_conv_bench.py on a B200 (1000 W), conv1 kernel / cuDNN: 18.5 / 9.4 us at 256 leaves, 19.1 / 17.1 at 768,
    # 19.4 / 23.9 at 1024, 27.8 / 31.1 at 2048, 46.6 / 58.0 at 4096.
    TRUNK_MIN_ROWS = 1024

    def __init__(self, model, engine, dtype=torch.bfloat16, use_stem=True, use_trunk=True, _buffers=True):
        self.engine, self.dtype = engine, dtype
        self._ctor = {"use_stem": use_stem, "use_trunk": use_trunk}
        dev = engine.device
        model = copy.deepcopy(model).to(dev).train(False)  # never move or retype the caller's (training) module
        rows, cols = engine.rows, engine.cols
        cap = engine.n_games * engine.max_pending
        self.stem = self.stem_mma = None
        c0 = model.conv0
        if use_stem and use_stem != "fma" and _stem_mma_ok(c0, engine, dtype):
            self.stem_mma = engine.nn_stem_mma_pack(_stem_mma_table(c0).to(dtype))      # r0 = relu(conv0(x) + b0), tensor cores
            self.stem_out = torch.empty((cap, rows, cols, c0.out_channels), dtype=dtype, device=dev) if _buffers else None
        elif use_stem and dtype in (torch.bfloat16, torch.float16) and (rows, cols) in ((4, 4), (6, 6), (3, 3), (5, 5)):
            ones = torch.ones(c0.out_channels, device=dev)
            self.stem = _stem_tables(c0, rows, cols) + (ones, torch.zeros_like(ones))  # the same on the CUDA cores
            self.stem_out = torch.empty((cap, rows, cols, c0.out_channels), dtype=dtype, device=dev) if _buffers else None
        else:
            self.conv0 = (_cl(c0.weight.detach(), dtype), c0.bias.detach().to(dtype), tuple(c0.padding))
        self.convs = []
        # The zero-padded convs (conv1-conv3) as the engine's tcgen05 trunk kernel (csrc/dbaz_trunk.cu) at batches of
        # TRUNK_MIN_ROWS and more: a GEMM per output position over its in-board taps with the z map and bias of the library
        # path, so no padding tap is multiplied and the result is the library's.  conv4 has no padding to skip and stays on cuDNN.
        convs = [getattr(model, f"conv{i}") for i in range(1, 5)]
        n_trunk = 0
        if (use_trunk and dtype == torch.bfloat16 and (self.stem_mma is not None or self.stem is not None) and c0.out_channels == 256
                and rows * cols <= 64):
            for c in convs:
                if (isinstance(c, nn.Sequential) or tuple(c.kernel_size) != (3, 3) or c.in_channels != 256 or c.out_channels != 256
                        or c.groups != 1 or tuple(c.stride) != (1, 1) or tuple(c.dilation) != (1, 1) or tuple(c.padding) != (1, 1)):
                    break
                n_trunk += 1
        self.trunk = [] if n_trunk else None
        # with the kernel, the library path (and its z maps) only serves batches below TRUNK_MIN_ROWS
        z_rows = min(cap, self.TRUNK_MIN_ROWS) if n_trunk else cap
        hw = (rows, cols)
        for i, conv in enumerate(convs, 1):
            s, t = _bn_affine(getattr(model, f"bn{i - 1}"))
            w32 = conv.weight.detach().float()
            pad = tuple(conv.padding)
            tmap = t.view(1, -1, 1, 1).expand(1, t.numel(), hw[0], hw[1]).contiguous()
            bpos = F.conv2d(tmap, w32, None, padding=pad)[0]  # image of the shift t under this conv, [cout, H', W']
            bias = conv.bias.detach().float()
            if i <= n_trunk:
                self.trunk.append((trunk_conv_pack(w32 * s.view(1, -1, 1, 1)),) + trunk_conv_bias(bias, bpos, pad[0]))
            z = None
            if pad == (0, 0):
                bias = bias + bpos[:, 0, 0]  # no padding: the same constant at every position
            else:
                z = bpos.to(dtype).unsqueeze(0).expand(z_rows, -1, -1, -1).contiguous(memory_format=torch.channels_last)
            self.convs.append((_cl(w32 * s.view(1, -1, 1, 1), dtype), bias.to(dtype), z, pad))
            hw = (bpos.shape[1], bpos.shape[2])
        self.trunk_plans = None
        if n_trunk and _buffers:
            # stem_out -> ping-pong NHWC buffers; the plans bind the buffers' full capacity once
            bufs = [torch.empty((cap, rows, cols, 256), dtype=dtype, device=dev) for _ in range(2)]
            x, self.trunk_plans = self.stem_out, []
            for i, (w, bp, b) in enumerate(self.trunk):
                self.trunk_plans.append(engine.nn_trunk_conv_plan(x, bufs[i % 2], w, bp, b, 1))
                x = bufs[i % 2]
            self.trunk_out = x
        c_out = N_CH_OUT(model)
        s, t = _bn_affine(model.bn4)
        # fc0 over the NHWC flatten of conv4's output, bn4 folded in (per channel, any position)
        w0 = model.fc0.weight.detach().float().view(-1, c_out, hw[0], hw[1])
        b0 = model.fc0.bias.detach().float() + (w0 * t.view(1, -1, 1, 1)).sum((1, 2, 3))
        w0 = (w0 * s.view(1, -1, 1, 1)).permute(0, 2, 3, 1).reshape(model.fc0.out_features, -1)
        s0, t0 = _bn_affine(model.bn_fc0)
        w1 = model.fc1.weight.detach().float()
        b1 = model.fc1.bias.detach().float() + w1 @ t0
        w1 = w1 * s0.view(1, -1)
        self.fcs = [(w0.to(dtype).t().contiguous(), b0.to(dtype)), (w1.to(dtype).t().contiguous(), b1.to(dtype))]
        s1, t1 = _bn_affine(model.bn_fc1)
        A = engine.A
        ld = (A + 1 + 7) // 8 * 8
        wh = torch.zeros((ld, model.policy_fc.in_features), dtype=torch.float32, device=dev)
        bh = torch.zeros((ld,), dtype=torch.float32, device=dev)
        wh[:A] = model.policy_fc.weight.detach(); wh[A] = model.value_fc.weight.detach()[0]
        bh[:A] = model.policy_fc.bias.detach(); bh[A] = model.value_fc.bias.detach()[0]
        bh = bh + wh @ t1
        wh = wh * s1.view(1, -1)
        self.wh, self.bh = wh.to(dtype).t().contiguous(), bh.to(dtype)
        # own kernels per batch: (stem,) (trunk convs at full batches,) heads
        self.engine_launches = (2 if (self.stem is not None or self.stem_mma is not None) else 1) + (len(self.trunk) if self.trunk else 0)
        engine.set_planes(dtype, channels_last=True)

    @torch.no_grad()
    def __call__(self, eng):
        n = eng.n_rows
        if self.stem_mma is not None:
            x = eng.nn_stem_mma(eng.leaf_states, self.stem_mma, self.stem_out[:n]).permute(0, 3, 1, 2)
        elif self.stem is not None:
            w01, bp, k2, s0, t0 = self.stem
            x = eng.nn_stem(eng.leaf_states, w01, bp, k2, s0, t0, self.stem_out[:n], mode=0).permute(0, 3, 1, 2)
        else:
            w, b, pad = self.conv0
            x = _conv_relu(eng.planes, w, b, pad)
        convs = self.convs
        if self.trunk is not None and n >= self.TRUNK_MIN_ROWS:
            for plan in self.trunk_plans:  # stem_out -> ping-pong buffers -> trunk_out, NHWC throughout
                eng.nn_trunk_conv(plan, n)
            x = self.trunk_out[:n].permute(0, 3, 1, 2)
            convs = convs[len(self.trunk_plans):]
        for w, b, z, pad in convs:
            x = _conv_relu(x, w, b, pad) if z is None else _conv_add_relu(x, w, z[:n], b, pad)
        x = x.permute(0, 2, 3, 1).reshape(n, -1)
        for w, b in self.fcs:
            x = torch._addmm_activation(b, x, w)  # relu(x @ w + b), ReLU in the GEMM epilogue
        eng.nn_heads(torch.addmm(self.bh, x, self.wh))


def N_CH_OUT(model):
    return model.conv4.out_channels


class FusedResNetZero(_ReloadablePlan):
    # Below this many leaves the library path is used even when the tower kernel is available: one tile through 41 stages
    # is a latency floor of ~190 us whatever the batch, cuDNN's 41 small kernels take 185-205 us at 64-168 leaves
    # (tools/tower_vs_cudnn.py on a B200: tower 0.87x at 64 leaves, 1.02x at 256, 1.35x at 1024, 2.3x at 2664, 1.76x at 15 984)
    TOWER_MIN_ROWS = 200

    """Inference plan for ResNetZero (nn.py:108-122).  Here BatchNorm sits between conv and ReLU, so it folds into
    the conv's own weights (per output channel) and bias, and every conv of the tower is ONE cuDNN kernel with its
    epilogue fused: conv-bias-ReLU for conv1 of a block, conv-add-bias-ReLU (z = the block input) for conv2 -- two
    kernels per residual block.  The input BatchNorm folds into the stem tables (leaf gather + conv0 + ReLU from the
    packed leaf states, own kernel); both 1x1 head convs are one conv, both head FCs one GEMM."""

    def __init__(self, model, engine, dtype=torch.bfloat16, use_stem=True, use_tower=True, _buffers=True):
        self.engine, self.dtype = engine, dtype
        self._ctor = {"use_stem": use_stem, "use_tower": use_tower}
        dev = engine.device
        model = copy.deepcopy(model).to(dev).train(False)  # never move or retype the caller's (training) module
        cap = engine.n_games * engine.max_pending

        def conv_fold(conv, bn):
            s, t = _bn_affine(bn)
            return conv.weight.detach().float() * s.view(-1, 1, 1, 1), conv.bias.detach().float() * s + t

        def conv_pack(conv, bn):
            if isinstance(conv, nn.Sequential):
                raise NotImplementedError("even kernel sizes are not supported by the fused plan")
            s, t = _bn_affine(bn)
            w = conv.weight.detach().float() * s.view(-1, 1, 1, 1)
            b = conv.bias.detach().float() * s + t
            return _cl(w, dtype), b.to(dtype), tuple(conv.padding)
        s_in, t_in = _bn_affine(model.bn_input)
        c0 = model.resnet.conv0
        self.fused_stem = self.stem_mma = None
        if use_stem and use_stem != "fma" and _stem_mma_ok(c0, engine, dtype):
            s0_, t0_ = _bn_affine(model.resnet.bn0)
            self.stem_mma = engine.nn_stem_mma_pack(_stem_mma_table(c0, s_in, t_in, s0_, t0_).to(dtype))  # relu(bn0(conv0(bn_input(x))))
            self.stem_out = torch.empty((cap, engine.rows, engine.cols, c0.out_channels), dtype=dtype, device=dev) if _buffers else None
        elif (use_stem and dtype in (torch.bfloat16, torch.float16) and not isinstance(c0, nn.Sequential) and tuple(c0.padding) == (1, 1)
                and c0.out_channels in (8, 16, 32, 64, 128, 256) and (engine.rows, engine.cols) in ((4, 4), (6, 6), (3, 3), (5, 5))):
            self.fused_stem = _stem_tables(c0, engine.rows, engine.cols, s_in, t_in) + _bn_affine(model.resnet.bn0)
            self.stem_out = torch.empty((cap, engine.rows, engine.cols, c0.out_channels), dtype=dtype, device=dev) if _buffers else None
        else:
            self.in_scale = s_in.view(1, -1, 1, 1).to(dtype)
            self.in_shift = t_in.view(1, -1, 1, 1).to(dtype)
            self.stem = conv_pack(c0, model.resnet.bn0)
        self.blocks = []
        for blk in model.resnet.resblocks:
            if blk.inner_conv is not None:
                raise NotImplementedError("inner_channels is not supported by the fused plan")
            self.blocks.append((conv_pack(blk.conv1, blk.bn1), conv_pack(blk.conv2, blk.bn2)))
        ph, vh = model.policy_head, model.value_head
        pw, pb, _ = conv_pack(ph.conv0, ph.bn0)
        vw, vb, _ = conv_pack(vh.conv0, vh.bn0)
        self.head_conv = (torch.cat([pw, vw], 0).contiguous(memory_format=torch.channels_last), torch.cat([pb, vb]))
        cp, cv = pw.shape[0], vw.shape[0]
        # The whole tower (every residual block) and the two 1x1 head convolutions as ONE persistent tcgen05 kernel
        # (csrc/dbaz_tower.cu): activations stay in shared memory across all convolutions, weights stream by TMA.
        self.tower = None
        blocks = list(model.resnet.resblocks)
        if (use_tower and self.stem_mma is not None and dtype == torch.bfloat16 and engine.tower_geometry()["ok"] and len(blocks) > 0
                and c0.out_channels == 64 and cp + cv in (16, 32)
                and all(tuple(c.kernel_size) == (3, 3) and tuple(c.padding) == (1, 1) and c.in_channels == 64 and c.out_channels == 64 and c.groups == 1
                        for b in blocks for c in (b.conv1, b.conv2))):
            folded = [conv_fold(c, bn) for b in blocks for c, bn in ((b.conv1, b.bn1), (b.conv2, b.bn2))]
            w3 = torch.stack([w for w, _ in folded])
            b3 = torch.stack([b for _, b in folded])
            pwf, pbf = conv_fold(ph.conv0, ph.bn0)
            vwf, vbf = conv_fold(vh.conv0, vh.bn0)
            packed, bias = tower_pack(w3, b3, torch.cat([pwf, vwf], 0).reshape(cp + cv, 64), torch.cat([pbf, vbf]))
            self.tower = (packed, bias, w3.shape[0], cp + cv)
            # one wave of the tower's persistent grid: the adaptive wave loop puts its batch sizes at multiples of it
            self.batch_quantum = engine.tower_geometry()["nb"] * engine.n_sms
            self.tower_tiles = engine.tower_tiles(cap) if _buffers else None
            self.tower_out = torch.empty((cap, engine.rows, engine.cols, cp + cv), dtype=dtype, device=dev) if _buffers else None
        hw = engine.rows * engine.cols
        A, fi = engine.A, vh.fc0.out_features
        # one GEMM over the NHWC-flattened [hw, cp+cv] head activations: columns [0, A) policy logits, [A, A+fi) value hidden
        W = torch.zeros((hw, cp + cv, A + fi), dtype=torch.float32, device=dev)
        W[:, :cp, :A] = ph.fc.weight.detach().view(A, cp, hw).permute(2, 1, 0)
        W[:, cp:, A:] = vh.fc0.weight.detach().view(fi, cv, hw).permute(2, 1, 0)
        self.head_w = W.reshape(hw * (cp + cv), A + fi).to(dtype).contiguous()
        self.head_b = torch.cat([ph.fc.bias.detach(), vh.fc0.bias.detach()]).to(dtype)
        self.v_w = vh.fc1.weight.detach().to(dtype).t().contiguous()
        self.v_b = vh.fc1.bias.detach().to(dtype)
        # fc1 of the value head finishes inside the heads kernel (Engine.nn_heads_mlp): weights then bias, float32
        self.v_wb = torch.cat([vh.fc1.weight.detach().float().reshape(-1), vh.fc1.bias.detach().float().reshape(-1)]).contiguous() if fi <= 32 else None
        self.fi = fi
        self.A = A
        self.ld = (A + 1 + 7) // 8 * 8
        self.logits = torch.zeros((cap, self.ld), dtype=dtype, device=dev) if _buffers else None
        self.engine_launches = (2 if (self.fused_stem is not None or self.stem_mma is not None) else 1) + (1 if self.tower is not None else 0)  # own kernels per batch: (stem,) (tower,) heads
        if self.tower is not None and _buffers:
            # the stem writes the tower's tiles; the NHWC stem output only serves the library path of tiny batches
            self.stem_out = torch.empty((min(cap, self.TOWER_MIN_ROWS), engine.rows, engine.cols, c0.out_channels), dtype=dtype, device=dev)
        engine.set_planes(dtype, channels_last=True)

    @torch.no_grad()
    def __call__(self, eng):
        n = eng.n_rows
        if self.tower is not None and n >= self.TOWER_MIN_ROWS:
            # stem -> tower -> heads: the stem writes the tower's planar tiles, no NHWC activation tensor in between
            packed, bias, n_stages, hc = self.tower
            eng.nn_stem_mma_tiles(eng.leaf_states, self.stem_mma, self.tower_tiles)
            h = eng.tower(self.tower_tiles, packed, bias, n_stages, hc, self.tower_out[:n]).reshape(n, -1)
            return self._heads(eng, h, n)
        if self.stem_mma is not None:
            x = eng.nn_stem_mma(eng.leaf_states, self.stem_mma, self.stem_out[:n]).permute(0, 3, 1, 2)
        elif self.fused_stem is not None:
            w01, bp, k2, s0, t0 = self.fused_stem
            x = eng.nn_stem(eng.leaf_states, w01, bp, k2, s0, t0, self.stem_out[:n], mode=1).permute(0, 3, 1, 2)
        else:
            w, b, pad = self.stem
            x = _conv_relu(eng.planes * self.in_scale + self.in_shift, w, b, pad)
        for (w1, b1, p1), (w2, b2, p2) in self.blocks:
            x = _conv_add_relu(_conv_relu(x, w1, b1, p1), w2, x, b2, p2)
        hw_, hb = self.head_conv
        h = _conv_relu(x, hw_, hb, (0, 0)).permute(0, 2, 3, 1).reshape(n, -1)
        return self._heads(eng, h, n)

    def _heads(self, eng, h, n):
        out = torch.addmm(self.head_b, h, self.head_w)
        if self.v_wb is not None:
            return eng.nn_heads_mlp(out, self.fi, self.v_wb)   # softmax + relu / fc1 / tanh of the value head in one kernel
        logits = self.logits[:n]
        logits[:, :self.A] = out[:, :self.A]
        logits[:, self.A:self.A + 1] = torch.addmm(self.v_b, F.relu(out[:, self.A:]), self.v_w)
        eng.nn_heads(logits)


def make_evaluator(model, engine, dtype=torch.bfloat16):
    """The fastest evaluator available for `model`: a fused inference plan for the two reference architectures,
    the plain module otherwise.  Plans snapshot (fold) the weights: build a new one after every training step."""
    from .dots_boxes.dots_boxes_nn import SimpleNN
    try:
        if isinstance(model, SimpleNN):
            return FusedSimpleNN(model, engine, dtype=dtype)
        if isinstance(model, ResNetZero):
            return FusedResNetZero(model, engine, dtype=dtype)
    except NotImplementedError:
        pass
    return DeviceEvaluator(model, engine, dtype=dtype)
