"""CPU restatements of the optimisers rebuild_optimisers can build (pixray.py:536-553) besides Adam, next to
oracle/ref_path.py's AdamState and with its interface: `State(z)` is a fresh instance (what every rebuild makes) and
`step(z, grad, lr)` returns the updated z.  The reference passes only lr, so every other hyper-parameter is the library
default.

Sources:
  AdamW    torch.optim.AdamW (torch 2.x, single-tensor path): weight_decay 0.01, betas 0.9 / 0.999, eps 1e-8
  Adagrad  torch.optim.Adagrad (torch 2.x): lr_decay 0, initial_accumulator_value 0, eps 1e-10
  Adamax   torch.optim.Adamax (torch 2.x, single-tensor path): betas 0.9 / 0.999, eps 1e-8
  DiffGrad torch_optimizer.DiffGrad 0.1.0 (pixray's requirements.txt:24): betas 0.9 / 0.999, eps 1e-8, weight_decay 0.
           torch_optimizer is not installed with this project, so this one is a transcription of the published
           algorithm, not checked against the library itself.
"""
import math

import torch

from oracle.ref_path import AdamState


class AdamWState(AdamState):
    """torch.optim.AdamW: z *= 1 - lr * weight_decay first, then exactly the Adam step."""

    def __init__(self, z, beta1=0.9, beta2=0.999, eps=1e-8, weight_decay=0.01):
        super().__init__(z, beta1, beta2, eps)
        self.wd = weight_decay

    def step(self, z, grad, lr):
        return super().step(z * (1 - lr * self.wd), grad, lr)


class AdagradState:
    """torch.optim.Adagrad: sum += g^2; z -= lr * g / (sqrt(sum) + eps)."""

    def __init__(self, z, eps=1e-10):
        self.s = torch.zeros_like(z)
        self.t = 0
        self.eps = eps

    def step(self, z, grad, lr):
        self.t += 1
        self.s.addcmul_(grad, grad, value=1)
        return z.addcdiv(grad, self.s.sqrt().add_(self.eps), value=-lr)


class AdamaxState:
    """torch.optim.Adamax: m.lerp_(g, 1 - b1); u = max(b2 u, |g| + eps); z -= lr / (1 - b1^t) * m / u."""

    def __init__(self, z, beta1=0.9, beta2=0.999, eps=1e-8):
        self.m = torch.zeros_like(z)
        self.u = torch.zeros_like(z)
        self.t = 0
        self.b1, self.b2, self.eps = beta1, beta2, eps

    def step(self, z, grad, lr):
        self.t += 1
        self.m.lerp_(grad, 1 - self.b1)
        self.u = torch.maximum(self.u * self.b2, grad.abs() + self.eps)
        return z.addcdiv(self.m, self.u, value=-lr / (1 - self.b1 ** self.t))


class DiffGradState:
    """torch_optimizer.DiffGrad 0.1.0: m, v as Adam; denom = sqrt(v) + eps (eps is not bias-corrected, unlike Adam);
    dfc = 1 / (1 + exp(-|p - g|)) with p the previous gradient (0 before the first step); p = g;
    z -= lr * sqrt(1 - b2^t) / (1 - b1^t) * (m * dfc) / denom."""

    def __init__(self, z, beta1=0.9, beta2=0.999, eps=1e-8):
        self.m = torch.zeros_like(z)
        self.v = torch.zeros_like(z)
        self.p = torch.zeros_like(z)
        self.t = 0
        self.b1, self.b2, self.eps = beta1, beta2, eps
        self.dfc = None  # the friction coefficient of the last step

    def step(self, z, grad, lr):
        self.t += 1
        self.m.mul_(self.b1).add_(grad, alpha=1 - self.b1)
        self.v.mul_(self.b2).addcmul_(grad, grad, value=1 - self.b2)
        denom = self.v.sqrt().add_(self.eps)
        bc1, bc2 = 1 - self.b1 ** self.t, 1 - self.b2 ** self.t
        self.dfc = torch.div(1.0, 1.0 + torch.exp(-(self.p - grad).abs()))
        self.p = grad.clone()
        step_size = lr * math.sqrt(bc2) / bc1
        return z.addcdiv(self.m * self.dfc, denom, value=-step_size)


STATES = {"Adam": AdamState, "AdamW": AdamWState, "Adagrad": AdagradState, "Adamax": AdamaxState,
          "DiffGrad": DiffGradState}
