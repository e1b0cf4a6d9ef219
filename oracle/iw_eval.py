"""Oracle (test infrastructure): CPU restatement of the reference's importance-weighted evaluation, on the same flat
`{parameter_name: tensor}` dict as oracle/model.py.

  log_p_x_given_z       sparse_vae/core/continuous_autoencoder.py:82-88 (p_of_x_given_z)
  estimate_log_prob_iw  sparse_vae/core/continuous_autoencoder.py:62-80, called by transformer_vae.py:71-79 (test_step)

Both take the latent samples z explicitly, so a GPU test can hand the oracle the very z the product drew.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.nn.functional as F

from . import model as omodel


def log_p_x_given_z(p: Dict[str, torch.Tensor], token_ids: torch.Tensor, z: torch.Tensor,
                    padding: Optional[torch.Tensor] = None, num_heads: int = 8, num_layers: int = 6, window: int = 4,
                    sparse: bool = True) -> torch.Tensor:
    """log p(x | z) per sequence [B]: teacher-forced `reconstruct` with the given z [B, 1, latent], fp32 log-softmax,
    column 0 set to 0 AFTER the softmax (padding tokens do not count), gathered at the next tokens and summed."""
    original = token_ids.long()
    padding = original.eq(0) if padding is None else padding
    x = F.embedding(original, p['input_layer.0.weight'])
    logits = omodel.reconstruct(p, x, z, padding, num_heads, num_layers, window, sparse)[..., :-1, :]
    log_probs = logits.float().log_softmax(dim=-1)
    log_probs[..., 0] = 0.0
    return log_probs.gather(dim=-1, index=original[..., 1:].unsqueeze(-1)).squeeze(-1).sum(dim=-1)


def posterior(p: Dict[str, torch.Tensor], token_ids: torch.Tensor, d_model: int,
              padding: Optional[torch.Tensor] = None) -> torch.distributions.Normal:
    """q(z | x) of the encoder (conditional_gaussian.py:18-30 without the KL): Normal(mu, exp(logvar / 2))."""
    original = token_ids.long()
    padding = original.eq(0) if padding is None else padding
    x = F.embedding(original, p['input_layer.0.weight'])
    enc = omodel.perceiver(p, x, padding, d_model)
    mu, logvar = omodel._linear(p, 'q_of_z_given_x.linear', enc).chunk(2, dim=-1)
    return torch.distributions.Normal(mu, logvar.exp().sqrt())


def estimate_log_prob_iw(p: Dict[str, torch.Tensor], token_ids: torch.Tensor, num_tokens: torch.Tensor, z: torch.Tensor,
                         d_model: int = 512, num_heads: int = 8, num_layers: int = 6, window: int = 4,
                         sparse: bool = True) -> dict:
    """Importance-weighted log p(x) with the given samples z [S, B, 1, latent] drawn from the encoder's posterior:
    logsumexp_s(log p(z_s) + log p(x | z_s) - log q(z_s | x)) - log S.  Returns dict(log_prob [B], the estimate;
    nll_iw, test_step's metric -mean_b(log_prob_b / num_tokens_b))."""
    q = posterior(p, token_ids, d_model)
    S = z.shape[0]
    log_p_z = (-0.5 * z.pow(2.0).sum(dim=-1) - math.log(math.sqrt(2 * math.pi)) * z.shape[-1]).reshape(S, -1)
    log_q_z = q.log_prob(z).sum(dim=-1).reshape(S, -1)
    log_p_x = torch.stack([log_p_x_given_z(p, token_ids, z[s], None, num_heads, num_layers, window, sparse)
                           for s in range(S)])
    log_prob = (log_p_z + log_p_x - log_q_z).logsumexp(dim=0) - math.log(S)
    return dict(log_prob=log_prob, nll_iw=-(log_prob / num_tokens).mean())
