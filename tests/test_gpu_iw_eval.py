"""GPU: importance-weighted NLL evaluation -- the `svae_vocab_logprob` kernel against fp64 and against the chain it
replaces (library GEMM + `svae_vocab_ce`), the fast `TransformerVAE.estimate_log_prob_iw` against the reference form
and the oracle, `Trainer.test` and the test.py script."""
import json
import math
import subprocess
import sys
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

sys.path.insert(0, str(Path(__file__).parent / 'golden'))
import make_golden as mg  # noqa: E402
from oracle import iw_eval as oiw  # noqa: E402

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


def _kernel(h, w, b, labels):
    from sparse_vae_b200 import _native as N
    rows, d = h.shape
    out = torch.empty(rows, device=h.device, dtype=torch.float32)
    N.check(N.lib.svae_vocab_logprob(h.data_ptr(), h.stride(0), w.data_ptr(), w.stride(0),
                                     b.data_ptr() if b is not None else None, N.svae_dtype(h.dtype), rows, w.shape[0], d,
                                     labels.data_ptr(), out.data_ptr(), N.current_stream(h.device)), 'svae_vocab_logprob')
    return out


def _inputs(rows, vocab, d, dtype, bias, seed=0):
    g = torch.Generator(device='cuda').manual_seed(seed)
    h = torch.randn(rows, d, device='cuda', generator=g).to(dtype)
    # logits of standard deviation ~1 (an LM head at initialisation).  The reference rounds the fp64 product, the kernel
    # its fp32 accumulation: near a rounding boundary the two differ by one 16-bit ulp, which moves the log-sum-exp by
    # (softmax weight of that logit) x ulp -- far inside the tolerance at this scale, but not for a spread of ~3, where
    # the largest logits (|x| ~ 12, bf16 ulp 0.0625) carry several percent of the softmax mass.
    w = (torch.randn(vocab, d, device='cuda', generator=g) / math.sqrt(d)).to(dtype)
    b = (torch.randn(vocab, device='cuda', generator=g) * 0.5).to(dtype) if bias else None
    labels = torch.randint(0, vocab, (rows,), device='cuda', generator=g)
    labels[::7] = 0
    labels[1::11] = vocab - 1
    return h, w, b, labels


def _ulp(x, dtype):
    mant = 7 if dtype == torch.bfloat16 else 10
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -14)))
    return torch.exp2(e - mant)


def _fp64_reference(h, w, b, labels, dtype):
    out = torch.empty(h.shape[0], dtype=torch.float64, device='cuda')
    x_lab = torch.empty_like(out)
    lse = torch.empty_like(out)
    for r0 in range(0, h.shape[0], 4096):
        r1 = min(h.shape[0], r0 + 4096)
        logits = h[r0:r1].double() @ w.double().T
        if b is not None:
            logits += b.double()
        logits = logits.to(dtype).double()
        lse[r0:r1] = torch.logsumexp(logits, dim=-1)
        x_lab[r0:r1] = logits.gather(1, labels[r0:r1, None]).squeeze(1)
    out = torch.where(labels == 0, torch.zeros_like(out), x_lab - lse)
    return out, x_lab, lse


def _check(got, ref, x_lab, lse, labels, dtype):
    tol = _ulp(x_lab, dtype) + 2e-5 * lse.abs()
    tol = torch.where(labels == 0, torch.zeros_like(tol), tol)
    err = (got.double() - ref).abs()
    bad = (err > tol).nonzero()
    assert bad.numel() == 0, f"{bad.numel()} rows out of tolerance, worst err {err.max().item():.3e}"
    assert err.mean().item() <= 1e-3
    assert torch.all(got[labels == 0] == 0)


@pytest.mark.parametrize('d', [256, 512])
@pytest.mark.parametrize('vocab', [8192, 24576, 32768])
@pytest.mark.parametrize('rows', [1, 127, 129, 1000, 16389])
def test_kernel_matches_fp64(rows, vocab, d):
    h, w, b, labels = _inputs(rows, vocab, d, torch.bfloat16, True, seed=rows + vocab + d)
    ref, x_lab, lse = _fp64_reference(h, w, b, labels, torch.bfloat16)
    _check(_kernel(h, w, b, labels), ref, x_lab, lse, labels, torch.bfloat16)


@pytest.mark.parametrize('bias', [False, True])
@pytest.mark.parametrize('dtype', [torch.bfloat16, torch.float16])
@pytest.mark.parametrize('d', [256, 512])
def test_kernel_dtypes_and_bias_match_fp64(dtype, bias, d):
    h, w, b, labels = _inputs(1000, 32768, d, dtype, bias, seed=3)
    ref, x_lab, lse = _fp64_reference(h, w, b, labels, dtype)
    _check(_kernel(h, w, b, labels), ref, x_lab, lse, labels, dtype)


def _chain(h, w, b, labels):
    from sparse_vae_b200 import _native as N
    rows = h.shape[0]
    nll = torch.empty(rows, device='cuda', dtype=torch.float32)
    weight = labels.ne(0).float()
    for r0 in range(0, rows, 16384):
        r1 = min(rows, r0 + 16384)
        logits = F.linear(h[r0:r1], w, b)
        N.check(N.lib.svae_vocab_ce(logits.data_ptr(), N.svae_dtype(h.dtype), r1 - r0, w.shape[0], logits.stride(0),
                                    labels[r0:r1].data_ptr(), weight[r0:r1].data_ptr(), nll[r0:r1].data_ptr(), 0,
                                    N.current_stream(h.device)), 'svae_vocab_ce')
    return torch.where(labels == 0, torch.zeros_like(nll), -nll)


@pytest.mark.parametrize('rows,dtype,bias', [(1000, torch.bfloat16, True), (16389, torch.float16, False),
                                             (65537, torch.bfloat16, True)])
def test_kernel_matches_gemm_plus_vocab_ce_chain(rows, dtype, bias):
    vocab, d = 32768, 512
    assert rows * vocab > 2 ** 31 or rows < 65537
    h, w, b, labels = _inputs(rows, vocab, d, dtype, bias, seed=11)
    want = _chain(h, w, b, labels)
    got = _kernel(h, w, b, labels)
    x_lab = torch.empty(rows, dtype=torch.float64, device='cuda')
    for r0 in range(0, rows, 16384):                  # the label logits of the chain (tolerance scale)
        r1 = min(rows, r0 + 16384)
        x_lab[r0:r1] = (h[r0:r1].float() * w[labels[r0:r1]].float()).sum(-1).double()
    lse = x_lab - want.double()
    _check(got, want.double(), x_lab, lse, labels, dtype)


def test_kernel_is_deterministic_and_rejects():
    from sparse_vae_b200.core.fused_ce import vocab_log_prob
    from sparse_vae_b200 import _native as N
    h, w, b, labels = _inputs(5000, 32768, 512, torch.bfloat16, True, seed=5)
    a, c = _kernel(h, w, b, labels), _kernel(h, w, b, labels)
    assert torch.equal(a, c)
    assert not N.lib.svae_vocab_logprob_supported(1000, 512, N.DTYPE_BF16)
    assert not N.lib.svae_vocab_logprob_supported(32768, 96, N.DTYPE_BF16)
    assert not N.lib.svae_vocab_logprob_supported(32768, 512, N.DTYPE_F32)
    lab = torch.ones(2, 7, dtype=torch.long, device='cuda')
    with torch.no_grad():
        head = torch.nn.Linear(512, 32768)
        with pytest.raises(ValueError):                                       # CPU tensors
            vocab_log_prob(torch.randn(2, 8, 512), head, lab.cpu())
        head = head.cuda()
        with pytest.raises(ValueError):                                       # fp32, no autocast
            vocab_log_prob(torch.randn(2, 8, 512, device='cuda'), head, lab)
        with torch.autocast('cuda', dtype=torch.bfloat16):
            with pytest.raises(ValueError):                                   # d = 96
                vocab_log_prob(torch.randn(2, 8, 96, device='cuda'), torch.nn.Linear(96, 32768).cuda(), lab)
            with pytest.raises(ValueError):                                   # vocab = 1000
                vocab_log_prob(torch.randn(2, 8, 512, device='cuda'), torch.nn.Linear(512, 1000).cuda(), lab)
            out = vocab_log_prob(torch.randn(2, 8, 512, device='cuda'), head, lab)
            assert out.shape == (2, 7) and out.dtype == torch.float32
    with torch.autocast('cuda', dtype=torch.bfloat16), pytest.raises(ValueError):
        vocab_log_prob(torch.randn(2, 8, 512, device='cuda', requires_grad=True), head, lab)


# ---------------------------------------------------------------- estimator ----------------------------------------
def _default_model():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    torch.manual_seed(7295)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams()))
    model.initialize_weights()
    return sv, model.cuda().eval()


def _padded_batch(sv, B, L, lengths, seed=1):
    from sparse_vae_b200.synthetic import synthetic_tokens, to_device
    return to_device(synthetic_tokens(B, L, seed=seed, lengths=lengths), torch.device('cuda'))


def _posterior_and_inputs(model, batch):
    from sparse_vae_b200.core.padded_tensor import split_padding
    tokens, padding = split_padding(batch['token_ids'])
    original = tokens.long()
    padding = original.eq(0) if padding is None else padding
    x = model.input_layer(original)
    return model.q_of_z_given_x(model.encoder(x, padding=padding)), x, original, padding


def _recording(q):
    drawn = []
    rsample = q.rsample
    q.rsample = lambda shape=torch.Size(): drawn.append(rsample(shape)) or drawn[-1]
    return drawn


@pytest.mark.parametrize('B,L,lengths,samples', [(2, 512, [512, 389], 8), (4, 1024, [1024, 1001, 700, 333], 4)])
def test_fast_estimator_matches_reference_form(B, L, lengths, samples):
    from sparse_vae_b200.core.continuous_autoencoder import ContinuousVAE
    sv, model = _default_model()
    batch = _padded_batch(sv, B, L, lengths)
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
        q, x, original, padding = _posterior_and_inputs(model, batch)
        drawn = _recording(q)
        torch.manual_seed(123)
        fast = model.estimate_log_prob_iw(q, x, original, samples, samples, padding=padding)
        drawn_fast = list(drawn)
        torch.manual_seed(123)
        ref = ContinuousVAE.estimate_log_prob_iw(model, q, x, original, samples, samples, padding=padding)
        drawn_ref = drawn[len(drawn_fast):]
    assert len(drawn_fast) == len(drawn_ref) == samples
    assert all(torch.equal(a, b) for a, b in zip(drawn_fast, drawn_ref))          # bit-identical z on both paths
    assert fast.shape == ref.shape == (B,)
    torch.testing.assert_close(fast, ref.float(), rtol=1e-3, atol=0)


@pytest.mark.parametrize('per_pass', [1, 64])
def test_samples_per_pass_agree_with_reference_form(per_pass):
    from sparse_vae_b200.core.continuous_autoencoder import ContinuousVAE
    sv, model = _default_model()
    batch = _padded_batch(sv, 2, 512, [512, 451], seed=2)
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
        q, x, original, padding = _posterior_and_inputs(model, batch)
        torch.manual_seed(9)
        fast = model.estimate_log_prob_iw(q, x, original, 64, 64, padding=padding, samples_per_pass=per_pass)
        torch.manual_seed(9)
        ref = ContinuousVAE.estimate_log_prob_iw(model, q, x, original, 64, 64, padding=padding)
    torch.testing.assert_close(fast, ref.float(), rtol=1e-3, atol=0)


def test_log_p_x_given_z_matches_oracle_c1():
    import sparse_vae_b200 as sv
    from sparse_vae_b200.core.lightning_shim import to_attrdict
    case = mg.MODEL_CASE
    hp = to_attrdict(sv.TransformerVAEHparams(d_model=case['d_model'], num_layers=case['num_layers'],
                                              num_heads=case['num_heads'], attn_window_size=case['window'],
                                              latent_depth=case['latent']))
    model = sv.TransformerVAE(hp)
    weights = mg.model_params([(n, tuple(p.shape)) for n, p in model.named_parameters()])
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(torch.tensor(weights[n]))
    model = model.cuda().eval()
    params = {n: t.detach().cpu().float() for n, t in model.state_dict().items()}
    tok = torch.tensor(mg.model_tokens(case))
    original = tok.long().cuda()
    padding = original.eq(0)
    z = torch.randn(case['B'], 1, case['latent'], generator=torch.Generator().manual_seed(4)) * 0.5
    want = oiw.log_p_x_given_z(params, tok, z, num_heads=case['num_heads'], num_layers=case['num_layers'],
                               window=case['window']).double()
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        with torch.no_grad():
            x = model.input_layer(original)
            fp32 = model.p_of_x_given_z(x, z.cuda(), original[..., 1:], padding=padding)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    with torch.no_grad():
        with torch.autocast('cuda', dtype=torch.bfloat16):
            x16 = model.input_layer(original)
            fast = model.log_p_x_given_z(x16, z.cuda()[None], original[..., 1:], padding)[0]
    assert torch.all((fp32.double().cpu() - want).abs() <= 1e-4 * want.abs())
    assert torch.all((fast.double().cpu() - want).abs() <= 1e-2 * want.abs())


def test_trainer_test_matches_direct_test_steps():
    from sparse_vae_b200.compat.lightning import Trainer
    from sparse_vae_b200.compat.refsurface import TextDataModule
    sv, model = _default_model()
    model.iw_samples = 4
    dm = TextDataModule(tokens_per_batch=2 * 512, seq_len=512, max_tokens_per_sample=512, num_batches=2)
    model.train()
    torch.manual_seed(31)
    results = Trainer(precision='bf16', gpus=1, logger=False).test(model, datamodule=dm, verbose=False)
    assert model.training
    nll = results[0]['nll_iw']
    assert math.isfinite(nll)
    model.eval()
    torch.manual_seed(31)
    vals, sizes = [], []
    with torch.no_grad(), torch.autocast('cuda', dtype=torch.bfloat16):
        for i, host in enumerate(dm.test_dataloader()):
            batch = {k: (v.to('cuda') if hasattr(v, 'to') else v) for k, v in host.items()}
            vals.append(float(model.test_step(batch, i)))
            sizes.append(batch['num_tokens'].shape[0])
    assert nll == pytest.approx(sum(v * n for v, n in zip(vals, sizes)) / sum(sizes), rel=1e-5)


def test_test_script_prints_one_json_line():
    r = subprocess.run([sys.executable, 'test.py', '--batch', '2', '--seq', '512', '--batches', '1', '--samples', '4'],
                       cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    out = json.loads(lines[0])
    assert math.isfinite(out['nll_iw']) and out['tokens'] == 1024
