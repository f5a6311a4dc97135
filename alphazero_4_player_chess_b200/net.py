"""The consumer of the encoded planes: a PyTorch policy/value network with the architecture of the
reference's `ResNet` (`src/py/net.py:6-63`: 3x3 conv stem, N residual blocks, policy head conv -> BN ->
ReLU -> Linear(A*R*R -> A*R*R), value head conv -> BN -> ReLU -> Linear -> tanh).  The network stays in
PyTorch by design (BASELINE.json north star); this module exists so that the self-play benchmark has
a random-init model of the named shape to drive.  It is not part of the hot path being replaced."""
from __future__ import annotations

import torch
from torch import nn

from .geometry import GEOMETRIES, NUM_STATE_CHANNELS


def _conv_bn_relu(cin: int, cout: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1), nn.BatchNorm2d(cout), nn.ReLU())


class _Residual(nn.Module):
    def __init__(self, ch: int):
        super().__init__()
        self.a = nn.Sequential(nn.Conv2d(ch, ch, 3, padding=1), nn.BatchNorm2d(ch), nn.ReLU(),
                               nn.Conv2d(ch, ch, 3, padding=1), nn.BatchNorm2d(ch))

    def forward(self, x):
        return torch.relu(self.a(x) + x)


class PolicyValueNet(nn.Module):
    def __init__(self, R: int, blocks: int = 10, hidden: int = 128, device: str | torch.device = "cuda"):
        super().__init__()
        g = GEOMETRIES[R]
        self.R = R
        self.device = torch.device(device)
        self.stem = _conv_bn_relu(NUM_STATE_CHANNELS, hidden)
        self.tower = nn.Sequential(*[_Residual(hidden) for _ in range(blocks)])
        self.policy = nn.Sequential(_conv_bn_relu(hidden, g.num_action_channels), nn.Flatten(),
                                    nn.Linear(g.action_space_size, g.action_space_size))
        self.value = nn.Sequential(_conv_bn_relu(hidden, NUM_STATE_CHANNELS), nn.Flatten(),
                                   nn.Linear(g.state_space_size, 1), nn.Tanh())
        self.to(self.device)

    def forward(self, x):
        x = self.tower(self.stem(x))
        return self.policy(x), self.value(x)


class InferenceNet:
    """Eval-mode inference view used inside the search loop (SURVEY 8f rank 1), same call contract as the reference's
    `self.neural_net(encoded)`: f32 planes in, f32 logits / values out.  The network stays PyTorch / cuDNN / cuBLAS --
    this only removes the passes over the activations that inference does not need:

      * BatchNorm (eval: running statistics) is folded into the preceding convolution's weights and bias, once;
      * convolution + bias + ReLU, and convolution + bias + residual + ReLU, each run as ONE cuDNN call
        (`torch.cudnn_convolution_relu` / `cudnn_convolution_add_relu`) in channels_last: 23 kernels for the 10-block
        tower instead of ~85;
      * the two heads' Linear weights have their input columns permuted from (c, h, w) to (h, w, c) order, so Flatten of
        the channels_last activation is a view instead of a transposing copy;
      * bf16=True: bf16 weights and activations (the 553 M-parameter policy Linear converted once, not per call);
        bf16=False: fp32 throughout = the reference's precision (`src/py/net.py` under PyTorch defaults).

    The wrapped module is left untouched (fp32, trainable); call refresh() after its weights change."""

    def __init__(self, net: PolicyValueNet, bf16: bool = True, fused: bool = True, split_policy_linear: bool = False):
        """split_policy_linear (fp32 only): the 23,520^2 policy Linear -- 1.13 TFLOP per 1,024 leaves, 17 of the 19.4 ms
        of the fp32 network on the SIMT pipes -- as a bf16 x 3 split product on the tensor cores: W = W1 + W2 + W3 and
        x = x1 + x2 + x3 in bf16 (24 mantissa bits each way), the six leading cross terms accumulated in fp32 inside
        three GEMMs.  Every bf16 product is exact in fp32; what remains is the tensor cores' fp32 accumulation, which is
        not IEEE round-to-nearest over K = 3 x 23,520: measured against an fp64 Linear on B200, strict fp32 is off by
        6e-7 of the logit scale, this split by 1.2e-5, TF32 and bf16 by orders of magnitude more
        (tests/test_gpu_mcts.py::test_split_policy_linear_matches_strict_fp32 prints the ladder).  An intermediate
        precision, NOT the reference's arithmetic: bench.py reports it beside the strict fp32 line, never instead."""
        self.dtype = torch.bfloat16 if bf16 else torch.float32
        self.module = net
        self.R, self.device = getattr(net, "R", None), net.device
        self.fused = bool(fused) and self.device.type == "cuda" and self._fused_ops_work()
        self.split = bool(split_policy_linear) and not bf16 and self.device.type == "cuda"
        self.refresh()

    # ---- weights ----------------------------------------------------------------------------------------
    @staticmethod
    def _fold(conv: nn.Conv2d, bn: nn.BatchNorm2d):
        """conv -> BN(eval) as one convolution: w * g / sqrt(var + eps), (b - mean) * g / sqrt(var + eps) + beta (fp32)."""
        scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        w = conv.weight.detach().float() * scale.view(-1, 1, 1, 1)
        b = (conv.bias.detach().float() - bn.running_mean.detach().float()) * scale + bn.bias.detach().float()
        return w, b

    def _conv(self, conv: nn.Conv2d, bn: nn.BatchNorm2d):
        w, b = self._fold(conv, bn)
        return (w.to(self.dtype).contiguous(memory_format=torch.channels_last), b.to(self.dtype).contiguous())

    def _head_linear(self, lin: nn.Linear, channels: int):
        out_f, in_f = lin.weight.shape
        w = lin.weight.detach().view(out_f, channels, in_f // channels).permute(0, 2, 1).reshape(out_f, in_f)
        return w.to(self.dtype).contiguous(), lin.bias.detach().to(self.dtype).contiguous()

    @torch.no_grad()
    def refresh(self) -> None:
        m = self.module
        self.stem = self._conv(m.stem[0], m.stem[1])
        self.tower = [(self._conv(r.a[0], r.a[1]), self._conv(r.a[3], r.a[4])) for r in m.tower]
        self.p_conv = self._conv(m.policy[0][0], m.policy[0][1])
        self.v_conv = self._conv(m.value[0][0], m.value[0][1])
        self.p_lin = self._head_linear(m.policy[2], m.policy[0][0].out_channels)
        self.v_lin = self._head_linear(m.value[2], m.value[0][0].out_channels)
        if self.split:
            w, parts = self.p_lin[0].float(), []
            for _ in range(3):
                part = w.to(torch.bfloat16)
                parts.append(part.t())
                w = w - part.float()
            self.p_split = torch.cat(parts, dim=0).contiguous()  # [3K, out]: rows W1^T | W2^T | W3^T
            self.p_lin = (None, self.p_lin[1])
            del w, parts

    def _fused_ops_work(self) -> bool:
        try:
            x = torch.zeros((1, 8, 4, 4), dtype=self.dtype, device=self.device).contiguous(memory_format=torch.channels_last)
            w = torch.zeros((8, 8, 3, 3), dtype=self.dtype, device=self.device).contiguous(memory_format=torch.channels_last)
            b = torch.zeros(8, dtype=self.dtype, device=self.device)
            y = torch.cudnn_convolution_relu(x, w, b, (1, 1), (1, 1), (1, 1), 1)
            torch.cudnn_convolution_add_relu(x, w, y, 1.0, b, (1, 1), (1, 1), (1, 1), 1)
            return True
        except Exception:
            return False

    # ---- forward ------------------------------------------------------------------------------------------
    def _conv_relu(self, x, wb):
        if self.fused:
            return torch.cudnn_convolution_relu(x, wb[0], wb[1], (1, 1), (1, 1), (1, 1), 1)
        return torch.relu_(torch.nn.functional.conv2d(x, wb[0], wb[1], padding=1))

    def _conv_add_relu(self, x, wb, residual):
        if self.fused:
            return torch.cudnn_convolution_add_relu(x, wb[0], residual, 1.0, wb[1], (1, 1), (1, 1), (1, 1), 1)
        return torch.relu_(torch.nn.functional.conv2d(x, wb[0], wb[1], padding=1).add_(residual))

    @torch.no_grad()
    def __call__(self, planes: torch.Tensor):
        n = planes.shape[0]
        x = planes.to(self.dtype).contiguous(memory_format=torch.channels_last)
        x = self._conv_relu(x, self.stem)
        for a, b in self.tower:
            x = self._conv_add_relu(self._conv_relu(x, a), b, x)
        p = self._conv_relu(x, self.p_conv).permute(0, 2, 3, 1).reshape(n, -1)  # (h, w, c) order: a view
        v = self._conv_relu(x, self.v_conv).permute(0, 2, 3, 1).reshape(n, -1)
        if self.split:
            K = p.shape[1]
            x1 = p.to(torch.bfloat16)
            r = p - x1.float()
            x2 = r.to(torch.bfloat16)
            x3 = (r - x2.float()).to(torch.bfloat16)
            logits = torch.mm(torch.cat([x1, x1, x1], dim=1), self.p_split, out_dtype=torch.float32)  # x1 (W1 + W2 + W3)
            logits += torch.mm(torch.cat([x2, x2], dim=1), self.p_split[: 2 * K], out_dtype=torch.float32)  # x2 (W1 + W2)
            logits += torch.mm(x3, self.p_split[:K], out_dtype=torch.float32)  # x3 W1
            logits += self.p_lin[1]
        else:
            logits = torch.nn.functional.linear(p, self.p_lin[0], self.p_lin[1])
        value = torch.tanh(torch.nn.functional.linear(v, self.v_lin[0], self.v_lin[1]))
        return logits.float(), value.float()


class AutocastNet:
    """Inference view of a model that is also being trained: eval-mode forward under bf16 autocast, weights
    untouched (fp32), f32 logits / values out."""

    def __init__(self, net: PolicyValueNet):
        self.net = net
        self.R, self.device = getattr(net, "R", None), net.device

    @torch.no_grad()
    def __call__(self, planes: torch.Tensor):
        was_training = self.net.training
        self.net.eval()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits, value = self.net(planes)
        self.net.train(was_training)
        return logits.float(), value.float()
