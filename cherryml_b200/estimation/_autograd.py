"""The fit behind torch's autograd: ``CherryLoss`` and ``RateMatrix``.

The reference's training loop is ordinary PyTorch: a ``RateMatrix`` module (``estimation/
_ratelearn/rate.py:31-188``) produces ``Q``, ``trainer.py:156-187`` evaluates
``-sum_k <C_k, log expm(t_k Q)>`` with ``torch.matrix_exp`` and lets autograd differentiate it,
``torch.optim.Adam`` steps.  ``CherryLoss.apply(Q, t, C)`` is that loss as ONE autograd node whose
forward and backward are the CUDA kernels of the fit (``cherry_fit_loss_grad``: batched
expm + fused ``C * log P`` reduction + the exact adjoint), so a reference-style loop

    model = RateMatrix(num_states=S, mode="pande_reversible", mask=mask, pi_requires_grad=True, initialization=Q0)
    opt = torch.optim.Adam(model.parameters(), lr=0.1)
    loss = CherryLoss.apply(model(), t, C) / C.sum();  loss.backward();  opt.step()

keeps working with the heavy part on the GPU.  (``quantized_transitions_mle`` does not go through
this node: it runs the whole epoch -- Q(theta), loss, gradient, Adam, best iterate -- in fused
kernels replayed from a CUDA graph.)
"""
from typing import Optional

import numpy as np
import torch

from ._engine import FitEngine, random_theta, theta_from_initialization

_ENGINES = {}


def _engine_for(t: torch.Tensor, C: torch.Tensor) -> FitEngine:
    """Device buffers / workspace for one (t, C) pair, created once per pair of tensors."""
    key = (C.data_ptr(), t.data_ptr(), tuple(C.shape), C.device.index, C._version, t._version)
    eng = _ENGINES.get(key)
    if eng is None:
        if len(_ENGINES) >= 4:
            _ENGINES.pop(next(iter(_ENGINES)))
        S = C.shape[-1]
        theta0 = random_theta(S)
        if C.dim() == 4:
            theta0 = np.tile(theta0, (C.shape[0], 1))
        eng = FitEngine(t.detach().cpu().numpy(), C.detach(), theta0, num_epochs=0, loss_normalization=False,
                        device=C.device)
        _ENGINES[key] = eng
    return eng


class CherryLoss(torch.autograd.Function):
    """``loss = -sum_k <C_k, log expm(t_k Q)>`` (per problem when ``Q`` is ``[P, S, S]``).

    ``Q``: fp64 CUDA tensor ``[S, S]`` or ``[P, S, S]``; ``t``: ``[K]`` or ``[P, K]``; ``C``:
    ``[K, S, S]`` or ``[P, K, S, S]`` (fp64, same device).  Returns a 0-dim tensor (or ``[P]``).
    The gradient flows to ``Q`` only."""

    @staticmethod
    def forward(ctx, Q: torch.Tensor, t: torch.Tensor, C: torch.Tensor) -> torch.Tensor:
        if not Q.is_cuda or Q.dtype != torch.float64:
            raise ValueError("CherryLoss needs an fp64 CUDA tensor Q (there is no CPU fallback)")
        eng = _engine_for(t, C)
        batched = Q.dim() == 3
        with torch.no_grad():
            eng.Q.copy_(Q.detach().reshape(eng.Q.shape))
        loss, grad = eng.loss_and_grad()
        ctx.save_for_backward(grad.clone() if batched else grad[0].clone())
        ctx.batched = batched
        return loss.clone() if batched else loss[0].clone()

    @staticmethod
    def backward(ctx, grad_out: torch.Tensor):
        (dQ,) = ctx.saved_tensors
        g = grad_out.view(-1, 1, 1) * dQ if ctx.batched else grad_out * dQ
        return g, None, None


class RateMatrix(torch.nn.Module):
    """``Q(theta)`` in the ``pande_reversible`` parameterisation with the reference module's
    arguments (``rate.py:31-188``): ``pi = softmax(pi_logits)``, ``S = softplus(upper)`` placed
    symmetrically off the diagonal (times the mask), ``Q = D^-1/2 S D^1/2`` with the diagonal set
    so that rows sum to zero.  Parameters are fp64 (the reference keeps fp32)."""

    def __init__(self, num_states: int, mode: str = "pande_reversible", mask=None, pi=None,
                 pi_requires_grad: bool = False, initialization: Optional[np.ndarray] = None,
                 device="cuda") -> None:
        super().__init__()
        if mode != "pande_reversible":
            raise NotImplementedError("only the pande_reversible parameterisation is implemented")
        S = int(num_states)
        self.num_states = S
        self.mode = mode
        if mask is None:
            m = np.ones((S, S))
        else:
            m = mask.detach().cpu().numpy() if isinstance(mask, torch.Tensor) else np.asarray(mask)
            m = m.astype(np.float64)
        if initialization is not None:
            theta = theta_from_initialization(np.asarray(initialization, dtype=np.float64), m)
        else:
            theta = random_theta(S)
        if pi is not None:
            p = pi.detach().cpu().numpy() if isinstance(pi, torch.Tensor) else np.asarray(pi)
            theta[:S] = np.log(p.astype(np.float64).reshape(-1))
        dev = torch.device(device)
        self._pi = torch.nn.Parameter(torch.tensor(theta[:S], dtype=torch.float64, device=dev),
                                      requires_grad=bool(pi_requires_grad))
        self.upper_diag = torch.nn.Parameter(torch.tensor(theta[S:], dtype=torch.float64, device=dev))
        iu = torch.triu_indices(S, S, offset=1, device=dev)
        self.register_buffer("_iu", iu)
        self.register_buffer("mask", torch.tensor(m, dtype=torch.float64, device=dev))

    def stationary_distribution(self) -> torch.Tensor:
        """``pi = softmax(pi_logits)``, the stationary distribution of ``forward()``'s rate matrix."""
        return torch.softmax(self._pi, dim=0)

    def forward(self) -> torch.Tensor:
        S = self.num_states
        pi = self.stationary_distribution()
        sym = torch.zeros((S, S), dtype=torch.float64, device=self.upper_diag.device)
        sym[self._iu[0], self._iu[1]] = torch.nn.functional.softplus(self.upper_diag)
        sym = (sym + sym.T) * self.mask
        sq = torch.sqrt(pi)
        off = sym * sq[None, :] / sq[:, None]
        return off - torch.diag(off.sum(dim=1))
