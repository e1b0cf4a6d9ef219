"""`TransformerVAE` (reference surface: sparse_vae/transformer_vae.py): Perceiver encoder -> fused Gaussian
bottleneck -> block-sparse causal decoder conditioned on z through per-layer projections that replace the first
position.  `training_step`, `reconstruct`, `sample`, `predict`, `test_step` keep the reference's signatures,
logged metrics and return values; state_dict keys are identical so reference checkpoints load."""
from __future__ import annotations

import math
from copy import deepcopy
from dataclasses import dataclass
from typing import Any, Dict, Optional

import torch
from torch import nn, Tensor
from torch.distributions.normal import Normal
from torch.utils.checkpoint import checkpoint

from .core.attention import Attention, Perceiver
from .core.conditional_gaussian import ConditionalGaussian
from .core.continuous_autoencoder import ContinuousVAE, ContinuousVAEHparams
from . import _native as N
from .core import decode, fused_ce
from .core.generation import GenerationState
from .core.lightning_shim import DictConfig
from .core.linear import WeightShadows
from .core.math_utils import marginal_kl
from .core.padded_tensor import split_padding
from .core.transformer_language_model import TransformerHparams, TransformerLanguageModel


class _ReplaceFirstPosition(torch.autograd.Function):
    """`torch.cat([row, x[..., 1:, :]], dim=-2)` evaluated IN PLACE on x (the reference's way of putting the latent
    at the [CLS] position of every decoder layer, transformer_vae.py:88): identical values, but no copy of the
    [B, L, d_model] activations in forward and one pass instead of zero-fill + copy in backward.  Only used when x is
    a temporary nobody else needs (the previous decoder layer's output)."""

    @staticmethod
    def forward(ctx, x: Tensor, row: Tensor):
        ctx.row_dtype = row.dtype
        x[..., :1, :] = row
        ctx.mark_dirty(x)
        return x

    @staticmethod
    def backward(ctx, g: Tensor):
        g_row = g[..., :1, :].to(ctx.row_dtype, copy=True)
        # The incoming gradient is the fresh output of the layer's first backward node (the LayerNorm fork) and has no
        # other reader, so its first row is cleared in place: a clone would copy [B, L, d_model] fp32 per decoder layer
        # (6 x 46 us per step).  Double backward keeps the out-of-place form.
        gx = g.clone() if (g.requires_grad or not g.is_contiguous()) else g
        gx[..., :1, :] = 0
        return gx, g_row


@dataclass
class TransformerVAEHparams(TransformerHparams, ContinuousVAEHparams):
    latent_depth: int = 64
    pretrained_encoder: bool = False
    pretrained_decoder: bool = False
    use_gpt2: bool = False
    early_stopping_metric: str = 'val_nll'


class TransformerVAE(TransformerLanguageModel, ContinuousVAE):
    # Decoder tokens per pass of the importance-weighted estimator's fast path: latent samples are stacked along the
    # batch so that each decoder forward covers about this many tokens (1 sample at 16 x 4096, 64 at 2 x 512).
    IW_TOKENS_PER_PASS = 65536
    # latent samples of test_step's importance-weighted estimate (the reference's fixed 100, one per rsample call)
    iw_samples: int = 100

    # `validate_args` of the posterior `Normal` returned by `training_step`.  None = torch's default, i.e. the reference's
    # behaviour: the constructor checks loc / scale on the HOST (`constraint.check(...).all()`), which synchronises the
    # device in the middle of every step and empties the launch queue.  A trainer that wants the CPU to run ahead of the
    # GPU sets this to False (bench.py does and says so in its `config`).
    validate_posterior: Optional[bool] = None

    def __init__(self, hparams: DictConfig):
        super().__init__(hparams)
        hp = self.hparams
        self.encoder_input_layer = deepcopy(self.input_layer)
        self.encoder_input_layer[0].weight = self.input_layer[0].weight
        self.q_of_z_given_x = ConditionalGaussian(hp.d_model, hp.latent_depth)
        self.encoder = Perceiver(num_layers=hp.num_layers // 2, num_latents=64, d_model=hp.d_model, bottleneck_width=1)
        self.z_projections = nn.ModuleList(nn.Linear(hp.latent_depth, hp.d_model) for _ in range(hp.num_layers))

    def training_step(self, batch: Dict[str, Tensor], batch_index: int, stage: str = 'train'):
        if (N.FUSED_EXTRAS and WeightShadows.ENABLED and self.device.type == 'cuda' and torch.is_autocast_enabled('cuda')
                and torch.is_grad_enabled()
                and torch.get_autocast_dtype('cuda') in (torch.bfloat16, torch.float16)):
            # one multi-tensor launch refreshes the 16-bit copies of all projection weights for this step
            shadows = self.__dict__.get('_weight_shadows')
            if shadows is None:
                shadows = self.__dict__['_weight_shadows'] = WeightShadows(self)
            with shadows.step():
                return self._training_step(batch, batch_index, stage)
        return self._training_step(batch, batch_index, stage)

    def _training_step(self, batch: Dict[str, Tensor], batch_index: int, stage: str = 'train'):
        tokens, padding = split_padding(batch['token_ids'])
        original = tokens.long()
        if padding is None:
            padding = original.eq(0)

        x = self.input_layer(original)
        encoder_out = self.encoder(x, padding=padding)
        z, kl, posterior = self.sample_z(encoder_out, token_counts=batch['num_tokens'], stage=stage)

        head = self.output_layer[-1]
        if fused_ce.supported(x, head) and not (stage == 'val' and hasattr(self, 'token_weights')):
            # vocabulary projection + cross-entropy without materialising the logits (core/fused_ce.py)
            hidden = self.reconstruct(x, z, padding=padding, return_hidden=True)
            nll = fused_ce.fused_vocab_nll(hidden, head, original[..., 1:])
            self.log(stage + '_nll', nll)
        else:
            logits = self.reconstruct(x, z, padding=padding)[..., :-1, :]
            nll = self.get_nll(logits, original[..., 1:], stage=stage,
                               bytes_per_token=batch['num_bytes'] / batch['num_tokens'] if stage == 'val' else None)
        loss = nll + self.hparams.kl_weight * kl

        if original.shape[0] > 1:
            self.log(stage + '_mc_mutual_info', kl - marginal_kl(posterior))

        if stage == 'train':
            return {'loss': loss, 'posterior': Normal(loc=posterior.loc.detach(), scale=posterior.scale.detach(),
                                                     validate_args=self.validate_posterior)}
        elif stage == 'val':
            self.log('val_loss', nll + kl)

    def validation_step(self, batch: Dict[str, Tensor], batch_index: int):
        return self.training_step(batch, batch_index, stage='val')

    def test_step(self, batch: Dict[str, Tensor], batch_index: int):
        tokens, padding = split_padding(batch['token_ids'])
        original = tokens.long()
        padding = original.eq(0) if padding is None else padding
        x = self.input_layer(original)
        posterior = self.q_of_z_given_x(self.encoder(x, padding=padding))
        log_prob = self.estimate_log_prob_iw(posterior, x, original, num_samples=self.iw_samples,
                                             num_iter=self.iw_samples, padding=padding) / batch['num_tokens']
        nll_iw = -log_prob.mean()
        self.log('nll_iw', nll_iw, on_step=True)
        return nll_iw

    def estimate_log_prob_iw(self, q_of_z: Normal, x: Tensor, labels: Tensor, num_samples: int, num_iter: int = 1,
                             padding: Tensor = None, samples_per_pass: Optional[int] = None):
        """Importance-weighted estimate of log p(x) per sequence (reference core/continuous_autoencoder.py:62-88).

        On the GPU under 16-bit autocast, without autograd and in eval mode, the latent samples are decoded in groups
        stacked along the batch (`samples_per_pass`, default: IW_TOKENS_PER_PASS decoder tokens per pass) and
        log p(x|z) comes from `fused_ce.vocab_log_prob`, so the [B, L, vocab] logits and their fp32 log-softmax are never
        allocated.  z is drawn exactly as the reference draws it (`num_iter` calls of `q_of_z.rsample([chunk])`), so
        both forms see the same samples (eval mode is required: training-mode dropout would draw from the generator
        between the reference's rsample calls).  Anything else runs the reference form
        (ContinuousVAE.estimate_log_prob_iw)."""
        head = self.output_layer[-1]
        x_raw, _ = split_padding(x)
        fast = (x_raw.is_cuda and torch.is_autocast_enabled('cuda') and not torch.is_grad_enabled() and not self.training
                and torch.get_autocast_dtype('cuda') in (torch.bfloat16, torch.float16)
                and fused_ce.vocab_log_prob_supported(x_raw, head))
        if not fast:
            return super().estimate_log_prob_iw(q_of_z, x, labels, num_samples, num_iter, padding)
        assert num_samples % num_iter == 0
        chunk = num_samples // num_iter
        zs, log_p_z, log_q_z = [], [], []
        for _ in range(num_iter):
            z = q_of_z.rsample([chunk])
            zs.append(z)
            log_p_z.append(self.prior_log_prob(z).reshape(chunk, -1))
            log_q_z.append(q_of_z.log_prob(z).sum(dim=-1).reshape(chunk, -1))
        log_p_x = self.log_p_x_given_z(x, torch.cat(zs), labels[..., 1:], padding, samples_per_pass)
        return (torch.cat(log_p_z) + log_p_x - torch.cat(log_q_z)).logsumexp(dim=0) - math.log(num_samples)

    def log_p_x_given_z(self, x: Tensor, z: Tensor, labels: Tensor, padding: Optional[Tensor] = None,
                        samples_per_pass: Optional[int] = None) -> Tensor:
        """log p(x | z_s) for latent samples z [S, B, 1, latent]: [S, B] fp32, the fast path of estimate_log_prob_iw
        (one decoder pass per group of samples stacked sample-major along the batch, `fused_ce.vocab_log_prob`)."""
        x, x_pad = split_padding(x)
        padding = x_pad if padding is None else padding
        S, B, L = z.shape[0], x.shape[0], x.shape[1]
        group = samples_per_pass or max(1, self.IW_TOKENS_PER_PASS // (B * L))
        out = []
        for s0 in range(0, S, group):
            g = min(group, S - s0)
            xg = x.repeat(g, 1, 1) if g > 1 else x
            pg = padding.repeat(g, 1) if (padding is not None and g > 1) else padding
            zg = z[s0:s0 + g].reshape(g * B, *z.shape[2:])
            hidden = self.reconstruct(xg, zg, padding=pg, return_hidden=True)
            lp = fused_ce.vocab_log_prob(hidden, self.output_layer[-1], labels.repeat(g, 1) if g > 1 else labels)
            out.append(lp.sum(dim=-1).reshape(g, B))
        return torch.cat(out)

    def predict(self, batch: Any, batch_idx: int = 0, dataloader_idx: Optional[int] = None):
        tokens, padding = split_padding(batch['token_ids'])
        original = tokens.long()
        padding = original.eq(0) if padding is None else padding
        return self.q_of_z_given_x(self.encoder(self.input_layer(original), padding=padding), get_kl=False)

    def reconstruct(self, x, z, padding: Optional[Tensor] = None, return_hidden: bool = False) -> Tensor:
        x, x_pad = split_padding(x)
        padding = x_pad if padding is None else padding
        use_checkpoint = self.hparams.grad_checkpointing and x.requires_grad
        for i, (layer, project) in enumerate(zip(self.decoder_layers, self.z_projections)):
            if N.FUSED_EXTRAS and x.is_cuda and x.requires_grad and not use_checkpoint:
                # layers > 0: x is the previous layer's own output, nobody else reads it; layer 0: the caller's
                # embedding must stay intact, so the row goes into a copy (a flat copy, not cat's strided gather)
                x = _ReplaceFirstPosition.apply(x if i > 0 and not x.is_leaf else x.clone(), project(z).to(x.dtype))
            else:
                x = torch.cat([project(z).to(x.dtype), x[..., 1:, :]], dim=-2)   # z takes the [CLS] position
            x = checkpoint(layer, x, None, padding, use_reentrant=False) if use_checkpoint else layer(x, padding=padding)
        if return_hidden:                                   # everything but the vocabulary projection
            return self.output_layer[:-1](x)
        return self.output_layer(x)

    def sample(self, max_length: int, batch_size: int = 1, **kwargs):
        if self.hparams.kl_weight < 1.0:        # unconditional samples are garbage before full KL weight
            return None
        with torch.autocast('cuda', enabled=self.device.type == 'cuda'):
            return self._sample(max_length, batch_size, **kwargs)

    def _sample(self, max_length: int, batch_size: int = 1, **kwargs):
        z = kwargs.pop('z', None)
        if z is None:
            z = torch.randn(batch_size, 1, self.hparams.latent_depth, device=self.device)

        state = GenerationState(max_length, batch_size, self.start_token, self.end_token, device=self.device, **kwargs)
        state.current_index = 1
        state.output_ids[:, 0] = self.start_token
        graphed = decode.supported(self, state)
        with Attention.kv_cache(max_length):
            while not state.should_stop():
                x = self.input_layer(state.prev_tokens())
                for layer, project in zip(self.decoder_layers, self.z_projections):
                    if state.current_index == 1:
                        x = torch.cat([project(z).to(x.dtype), x[..., 1:, :]], dim=-2)
                    x = layer(x)
                Attention.update_kv_cache(state.process_logits(self.output_layer(x.squeeze(1))))
                if graphed:                 # position 0 (the z row) is done; every later token is one graph replay
                    decode.GraphedDecoder(self, state, decode.TRACE).run()
                    break
        return state.final_output()
