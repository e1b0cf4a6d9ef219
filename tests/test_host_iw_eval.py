"""CPU: the loop logic of the compat `Trainer.test`, the held-out data stream, the rejects of `vocab_log_prob` and the
internal consistency of the importance-weighted oracle (oracle/iw_eval.py)."""
import math

import pytest
import torch
from torch import nn

from oracle import iw_eval as oiw
from oracle import model as omodel


def _tiny_dense_lm():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    hp = to_attrdict(sv.TransformerHparams(d_model=32, num_heads=2, num_layers=2,
                                           sparse_self_attention=False))
    torch.manual_seed(0)
    model = sv.TransformerLanguageModel(hp)
    model.initialize_weights()
    return model


def _batches(n, B, L, vocab=2 ** 15):
    g = torch.Generator().manual_seed(11)
    out = []
    for i in range(n):
        tok = torch.randint(3, vocab, (B + i, L), generator=g)          # different batch sizes: a weighted mean
        tok[:, 0] = 1
        tok[-1, L - 3:] = 0
        counts = tok.ne(0).sum(-1)
        out.append({'token_ids': tok, 'num_tokens': counts, 'num_bytes': 4 * counts})
    return out


def test_trainer_test_cpu_weighted_mean_and_mode_restored():
    from sparse_vae_b200.compat.lightning import Trainer
    model = _tiny_dense_lm()
    batches = _batches(3, 2, 16)
    model.train()
    results = Trainer(precision=32, logger=False).test(model, test_dataloaders=[batches], verbose=False)
    assert model.training
    assert isinstance(results, list) and len(results) == 1 and 'val_nll' in results[0]
    model.eval()
    num, den = 0.0, 0
    with torch.no_grad():
        for i, b in enumerate(batches):
            model.logged.clear()
            model.test_step(b, i)
            num += float(model.logged['val_nll']) * b['token_ids'].shape[0]
            den += b['token_ids'].shape[0]
    assert math.isfinite(results[0]['val_nll'])
    assert results[0]['val_nll'] == pytest.approx(num / den, rel=1e-6)


def test_trainer_test_leaves_eval_mode_and_loads_checkpoint(tmp_path):
    from sparse_vae_b200.compat.lightning import Trainer
    model = _tiny_dense_lm()
    ckpt = tmp_path / 'w.ckpt'
    torch.save({'state_dict': model.state_dict()}, ckpt)
    with torch.no_grad():
        for p in model.parameters():
            p.add_(1.0)
    model.eval()
    batches = _batches(1, 2, 16)
    r = Trainer(logger=False).test(model, test_dataloaders=[batches], ckpt_path=str(ckpt), verbose=False)
    assert not model.training
    fresh = _tiny_dense_lm()
    fresh.eval()
    with torch.no_grad():
        fresh.test_step(batches[0], 0)
    assert r[0]['val_nll'] == pytest.approx(float(fresh.logged['val_nll']), rel=1e-6)


def test_test_dataloader_is_a_disjoint_stream():
    from sparse_vae_b200.compat.refsurface import TextDataModule
    dm = TextDataModule(tokens_per_batch=2 * 64, seq_len=64, max_tokens_per_sample=64, num_batches=2)
    first = lambda it: next(iter(it))['token_ids'].as_raw()          # noqa: E731
    test, train, val = first(dm.test_dataloader()), first(dm.train_dataloader()), first(dm.val_dataloader())
    assert test.shape == train.shape == (2, 64)
    assert not torch.equal(test, train) and not torch.equal(test, val)
    assert torch.equal(test, first(dm.test_dataloader()))                # reproducible


def test_vocab_log_prob_rejects_cpu_and_grad():
    from sparse_vae_b200.core.fused_ce import vocab_log_prob
    head = nn.Linear(512, 32768)
    h = torch.randn(1, 4, 512)
    labels = torch.ones(1, 3, dtype=torch.long)
    with torch.no_grad(), pytest.raises(ValueError):
        vocab_log_prob(h, head, labels)                                   # CPU tensors
    with pytest.raises(ValueError):
        vocab_log_prob(h, head, labels)                                   # the head requires grad
    with torch.no_grad(), pytest.raises(ValueError):
        vocab_log_prob(h, head, labels[:, :2])                            # labels not shifted by one


def test_oracle_iw_single_sample_is_the_importance_weight():
    p = {k: v.detach() for k, v in omodel.init_params(d_model=64, num_layers=2, latent=8, vocab=256, seed=3).items()}
    g = torch.Generator().manual_seed(5)
    tok = torch.randint(3, 256, (2, 64), generator=g)
    tok[:, 0] = 1
    tok[1, 50:] = 0
    counts = tok.ne(0).sum(-1)
    q = oiw.posterior(p, tok, 64)
    z = q.sample([1])
    kw = dict(num_heads=1, num_layers=2, window=4)
    lp = oiw.log_p_x_given_z(p, tok, z[0], **kw)
    out = oiw.estimate_log_prob_iw(p, tok, counts, z, d_model=64, **kw)
    log_w = (-0.5 * z.pow(2).sum(-1) - 0.5 * math.log(2 * math.pi) * 8).reshape(1, -1) + lp - q.log_prob(z).sum(-1).reshape(1, -1)
    torch.testing.assert_close(out['log_prob'], log_w[0], rtol=1e-6, atol=1e-4)
    assert torch.isfinite(out['nll_iw'])
    # padding tokens contribute 0: the padded sequence's log p(x|z) equals the sum over its real next tokens only
    logits = omodel.reconstruct(p, torch.nn.functional.embedding(tok, p['input_layer.0.weight']), z[0], tok.eq(0),
                                1, 2, 4)[..., :-1, :].log_softmax(-1)
    manual = logits[1, :49].gather(-1, tok[1, 1:50, None]).sum()
    torch.testing.assert_close(lp[1], manual, rtol=1e-6, atol=1e-4)


@pytest.mark.reference
def test_oracle_iw_matches_reference_estimate_log_prob_iw():
    """The oracle against the reference's own `estimate_log_prob_iw` on the same z (recorded from its rsample calls)."""
    import sys
    from pathlib import Path
    from oracle import reference_harness as rh
    sys.path.insert(0, str(Path(__file__).parent / 'golden'))
    import make_golden as mg
    ref = rh.load_reference()
    case = mg.MODEL_CASE
    hp = rh.default_hparams(d_model=case['d_model'], num_layers=case['num_layers'], num_heads=case['num_heads'],
                            attn_window_size=case['window'], latent_depth=case['latent'])
    model = ref.transformer_vae.TransformerVAE(hp)
    weights = mg.model_params([(n, tuple(p.shape)) for n, p in model.named_parameters()])
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(torch.tensor(weights[n]))
    model.eval()
    tok = torch.tensor(mg.model_tokens(case))
    original = tok.long()
    padding = original.eq(0)
    counts = torch.tensor(case['lengths'])
    p = {n: t.detach().float() for n, t in model.state_dict().items()}
    with torch.no_grad():
        x = model.input_layer(original)
        q = model.q_of_z_given_x(model.encoder(x, padding=padding))
        q = q[-1] if isinstance(q, tuple) else q
        drawn = []
        rsample = q.rsample
        q.rsample = lambda shape=torch.Size(): drawn.append(rsample(shape)) or drawn[-1]
        torch.manual_seed(7295)
        got = model.estimate_log_prob_iw(q, x, original, num_samples=4, num_iter=4, padding=padding)
    z = torch.cat(drawn)
    want = oiw.estimate_log_prob_iw(p, tok, counts, z, d_model=case['d_model'], num_heads=case['num_heads'],
                                    num_layers=case['num_layers'], window=case['window'])
    torch.testing.assert_close(want['log_prob'], got.float(), rtol=1e-4, atol=1e-2)
