"""Generates the golden fixtures in this directory by running the UNMODIFIED reference
(a checkout of norabelrose/sparse-vae, imported behind the stubs of oracle/reference_harness.py) on CPU in fp32.

Run with that checkout named:   SPARSE_VAE_REFERENCE=<checkout> python tests/golden/make_golden.py
The fixtures are committed; tests read the .npz files and never touch the reference.

Inputs are produced with numpy's legacy `RandomState` (bit-stable across numpy versions) so that only
the reference's OUTPUTS need to be stored.  Seed 7295 is the reference's own (train.py:15).
"""
from __future__ import annotations

import hashlib
import sys
import zlib
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

from oracle import reference_harness as rh  # noqa: E402

OUT = Path(__file__).resolve().parent
SEED = 7295


# ----------------------------------------------------------------------------- shared input recipes
def attention_inputs(case: dict):
    """q, k, v, dout [B,H,L,Dh] fp32 and an optional bool padding mask, from RandomState(case seed)."""
    rs = np.random.RandomState(case['seed'])
    shp = (case['B'], case['H'], case['L'], case['Dh'])
    q, k, v, dout = (rs.standard_normal(shp).astype(np.float32) for _ in range(4))
    pad = None
    if case.get('lengths') is not None:
        pad = np.zeros((case['B'], case['L']), dtype=np.bool_)
        for b, n in enumerate(case['lengths']):
            pad[b, n:] = True
    return q, k, v, dout, pad


ATTENTION_CASES = [
    dict(name='causal_cls_w4', seed=SEED + 1, B=2, H=2, L=256, Dh=32, window=4, causal=True, include_cls=True,
         lengths=[256, 201]),
    dict(name='causal_cls_w2_dh64', seed=SEED + 2, B=1, H=2, L=160, Dh=64, window=2, causal=True, include_cls=True,
         lengths=None),
    dict(name='bidir_nocls_w4', seed=SEED + 3, B=1, H=2, L=192, Dh=32, window=4, causal=False, include_cls=False,
         lengths=[150]),
    dict(name='causal_nocls_w3', seed=SEED + 4, B=1, H=2, L=128, Dh=16, window=3, causal=True, include_cls=False,
         lengths=None),
    dict(name='bidir_cls_w5', seed=SEED + 5, B=1, H=2, L=224, Dh=32, window=5, causal=False, include_cls=True,
         lengths=None),
]

LAYOUT_CASES = [(nb, w, causal, cls)
                for nb in (1, 2, 3, 4, 5, 8, 16, 17, 128)
                for w in (1, 2, 3, 4, 5, 6, 8)
                for causal in (True, False)
                for cls in (True, False)]


def model_params(named_shapes, seed=SEED):
    """Deterministic weights keyed by parameter NAME (independent of construction order)."""
    out = {}
    for name, shape in named_shapes:
        rs = np.random.RandomState((zlib.crc32(name.encode()) + seed) % (2 ** 31))
        if name.endswith('layer_norm.weight') or name == 'output_layer.2.weight':
            w = 1.0 + 0.05 * rs.standard_normal(shape)
        elif name.endswith('.bias'):
            w = 0.02 * rs.standard_normal(shape)
        elif name.endswith('learned_queries'):
            w = rs.standard_normal(shape)
        else:
            w = 0.02 * rs.standard_normal(shape)
        out[name] = w.astype(np.float32)
    return out


MODEL_CASE = dict(B=2, L=512, d_model=256, num_layers=4, num_heads=8, window=4, latent=64,
                  lengths=[512, 389], seed=SEED + 10)


def model_tokens(case):
    rs = np.random.RandomState(case['seed'])
    tok = rs.randint(3, 2 ** 15, size=(case['B'], case['L'])).astype(np.int64)
    tok[:, 0] = 1                                    # [CLS]
    for b, n in enumerate(case['lengths']):
        tok[b, n - 1] = 2                            # [SEP]
        tok[b, n:] = 0                               # padding
    return tok


# ----------------------------------------------------------------------------- generators
def gen_layouts(ref):
    SA = ref.core.SparseAttention
    packed, meta = {}, []
    for i, (nb, w, causal, cls) in enumerate(LAYOUT_CASES):
        sa = SA(window_size=w, causal=causal, include_cls=cls, num_heads=2, max_seq_len=32 * 160)
        lay = sa.get_master_layout()[..., :nb, :nb]
        assert lay.dtype == torch.int64 and (lay[0] == lay[1]).all()
        packed[f'l{i}'] = np.packbits(lay[0].numpy().astype(np.uint8))
        meta.append((nb, w, int(causal), int(cls), int(lay[0].sum())))
    # full-size master layout facts (max_seq_len 115200 -> 3600 blocks), stored as digests
    big = []
    for w in (4, 6, 8):
        sa = SA(window_size=w)
        m = sa.get_master_layout()
        for nb in (512, 3600):
            sl = m[0, :nb, :nb].contiguous().numpy()
            big.append((w, nb, int(sl.sum()), hashlib.sha256(sl.astype(np.uint8).tobytes()).hexdigest()))
        assert tuple(m.shape) == (8, 3600, 3600)
    np.savez_compressed(OUT / 'layout_golden.npz', meta=np.asarray(meta, dtype=np.int64),
                        big=np.asarray(big, dtype=object).astype(str), **packed)


def attention_rows(case):
    """The sequence positions whose rows of out / dq / dk / dv are stored: a seeded three quarters of them, which keeps
    attention_golden.npz under 1 MB."""
    L = case['L']
    return np.sort(np.random.RandomState(case['seed']).choice(L, 3 * L // 4, replace=False))


def gen_attention(ref):
    SA = ref.core.SparseAttention
    store = {}
    for case in ATTENTION_CASES:
        q, k, v, dout, pad = attention_inputs(case)
        qt, kt, vt = (torch.tensor(t, requires_grad=True) for t in (q, k, v))
        sa = SA(window_size=case['window'], causal=case['causal'], include_cls=case['include_cls'],
                num_heads=case['H'], max_seq_len=32 * 64)
        kpm = torch.tensor(pad) * -1e7 if pad is not None else None        # core/attention.py:79
        out = sa(qt, kt, vt, key_padding_mask=kpm)                          # the reference's own __call__
        out.backward(torch.tensor(dout))
        rows = attention_rows(case)
        store[f"{case['name']}.rows"] = rows
        for nm, t in (('out', out), ('dq', qt.grad), ('dk', kt.grad), ('dv', vt.grad)):
            store[f"{case['name']}.{nm}"] = t.detach().numpy().astype(np.float32)[:, :, rows]
    np.savez_compressed(OUT / 'attention_golden.npz', **store)


def gen_bottleneck(ref):
    """ConditionalGaussian + ContinuousVAE.sample_z of the reference on CPU (fp32)."""
    rs = np.random.RandomState(SEED + 20)
    B, D, latent = 5, 96, 64
    enc = rs.standard_normal((B, 1, D)).astype(np.float32)
    W = (0.3 * rs.standard_normal((2 * latent, D))).astype(np.float32)
    bias = (0.1 * rs.standard_normal((2 * latent,))).astype(np.float32)
    counts = np.asarray([512, 389, 77, 1024, 33], dtype=np.int64)

    cg = ref.core.ConditionalGaussian(D, latent)
    with torch.no_grad():
        cg.linear.weight.copy_(torch.tensor(W))
        cg.linear.bias.copy_(torch.tensor(bias))

    class Host(ref.core.ContinuousVAE):          # sample_z only needs q_of_z_given_x and self.log
        def __init__(self):
            torch.nn.Module.__init__(self)
            self.logged = {}
            self.q_of_z_given_x = cg

        def reconstruct(self, x, z):
            raise NotImplementedError

    host = Host()
    x = torch.tensor(enc, requires_grad=True)
    torch.manual_seed(SEED)
    z, kl, q_of_z = host.sample_z(x, torch.tensor(counts))
    torch.manual_seed(SEED)
    eps = torch.empty(B, 1, latent).normal_()                      # the noise rsample() just drew
    dz = torch.tensor(rs.standard_normal((B, 1, latent)).astype(np.float32))
    dkl = 0.7
    mulogvar = cg.linear(x)
    gz, = torch.autograd.grad([z, kl], [x], [dz, torch.tensor(dkl)], retain_graph=True)
    # gradient w.r.t. the Linear output, recomputed through the reference module
    ml = mulogvar.detach().requires_grad_(True)
    mu, logvar = ml.chunk(2, dim=-1)
    var = logvar.exp()
    z2 = mu + eps * var.sqrt()
    kl2 = (0.5 * (mu ** 2 + var - logvar - 1.0)).flatten(1).sum(-1).div(torch.tensor(counts)).mean()
    assert torch.equal(z2, z) and torch.allclose(kl2, kl)
    gml, = torch.autograd.grad([z2, kl2], [ml], [dz, torch.tensor(dkl)])
    _, kl_elem = cg(x, get_kl=True)
    np.savez_compressed(
        OUT / 'bottleneck_golden.npz', enc=enc, W=W, bias=bias, counts=counts, eps=eps.numpy(),
        z=z.detach().numpy(), kl=kl.detach().numpy(), raw_kl=host.logged['train_kl'].numpy(),
        kl_elem=kl_elem.detach().numpy(), sigma=q_of_z.scale.detach().numpy(), loc=q_of_z.loc.detach().numpy(),
        mulogvar=mulogvar.detach().numpy(), dz=dz.numpy(), dkl=np.float32(dkl), d_enc=gz.numpy(),
        d_mulogvar=gml.numpy())


def gen_model(ref):
    """BASELINE config 1: one TransformerVAE.training_step + backward (dropout off via eval())."""
    case = MODEL_CASE
    hp = rh.default_hparams(d_model=case['d_model'], num_layers=case['num_layers'], num_heads=case['num_heads'],
                            attn_window_size=case['window'], latent_depth=case['latent'])
    model = ref.transformer_vae.TransformerVAE(hp)
    named = [(n, tuple(p.shape)) for n, p in model.named_parameters()]
    weights = model_params(named)
    with torch.no_grad():
        for n, p in model.named_parameters():
            p.copy_(torch.tensor(weights[n]))
    model.eval()                                   # Dropout(0.1) off; nothing else depends on the mode
    tok = model_tokens(case)
    PT = ref.core.PaddedTensor
    lengths = torch.tensor(case['lengths'])
    batch = {'token_ids': PT.from_raw(torch.tensor(tok)), 'num_tokens': lengths, 'num_bytes': 4 * lengths}
    torch.manual_seed(SEED)
    out = model.training_step(batch, 0)
    torch.manual_seed(SEED)
    eps = torch.empty(case['B'], 1, case['latent']).normal_()
    loss = out['loss']
    loss.backward()
    grads = {n: p.grad for n, p in model.named_parameters()}
    no_grad = sorted(n for n, g in grads.items() if g is None)
    gnorm = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values() if g is not None))
    keep = ['q_of_z_given_x.linear.bias', 'z_projections.0.bias', 'decoder_layers.0.attention.q_linear.bias',
            'decoder_layers.3.attention.v_linear.bias', 'encoder.first_layer.attention.k_linear.bias',
            'decoder_layers.1.ffn.0.bias', 'output_layer.3.bias']
    store = {('grad.' + n): grads[n].numpy() for n in keep}
    np.savez_compressed(
        OUT / 'model_golden.npz', eps=eps.numpy(), loss=np.float64(loss.item()),
        nll=np.float64(model.logged['train_nll'].item()), raw_kl_mean=np.float64(model.logged['train_kl'].item()),
        grad_norm=np.float64(gnorm.item()), no_grad=np.asarray(no_grad),
        param_names=np.asarray([n for n, _ in named]),
        param_shapes=np.asarray([','.join(map(str, s)) for _, s in named]),
        posterior_loc=out['posterior'].loc.numpy(), posterior_scale=out['posterior'].scale.numpy(), **store)


if __name__ == '__main__':
    ref = rh.load_reference()
    gen_layouts(ref)
    gen_attention(ref)
    gen_bottleneck(ref)
    gen_model(ref)
    for f in sorted(OUT.glob('*.npz')):
        print(f.name, f.stat().st_size)
