#!/usr/bin/env python
"""`python test.py [checkpoint] [--batch B] [--seq L] [--batches N] [--samples S] [--precision bf16|16]`

Evaluates the importance-weighted NLL bound (`nll_iw`, TransformerVAE.test_step with S latent samples per sequence)
on held-out synthetic batches through `Trainer.test`, like the reference's test.py.  Random-init weights unless a
state_dict / Lightning checkpoint path is given (reference checkpoints load: the parameter names are identical).
Prints one JSON line: nll_iw, tokens evaluated, wall seconds."""
import argparse
import json
import time

import torch

import sparse_vae_b200 as sv
from sparse_vae_b200.compat.lightning import Trainer
from sparse_vae_b200.compat.refsurface import TextDataModule
from sparse_vae_b200.core.lightning_shim import to_attrdict


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument('checkpoint', nargs='?', default=None)
    ap.add_argument('--batch', type=int, default=16)
    ap.add_argument('--seq', type=int, default=4096)
    ap.add_argument('--batches', type=int, default=1)
    ap.add_argument('--samples', type=int, default=100)
    ap.add_argument('--precision', choices=('bf16', '16'), default='bf16')
    args = ap.parse_args(argv)

    torch.manual_seed(7295)
    model = sv.TransformerVAE(to_attrdict(sv.TransformerVAEHparams()))
    model.initialize_weights()
    if args.checkpoint:
        state = torch.load(args.checkpoint, map_location='cpu', weights_only=False)
        model.load_state_dict(state.get('state_dict', state))
    model.iw_samples = args.samples
    data = TextDataModule(tokens_per_batch=args.batch * args.seq, seq_len=args.seq, max_tokens_per_sample=args.seq,
                          num_batches=args.batches)
    trainer = Trainer(precision=args.precision, gpus=1, logger=False)
    model.to(trainer._device())
    if trainer._device().type == 'cuda':
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    results = trainer.test(model, datamodule=data, verbose=False)
    if trainer._device().type == 'cuda':
        torch.cuda.synchronize()
    seconds = time.perf_counter() - t0
    print(json.dumps({'nll_iw': results[0].get('nll_iw'), 'tokens': args.batch * args.seq * args.batches,
                      'samples': args.samples, 'precision': args.precision, 'seconds': round(seconds, 3)}))


if __name__ == '__main__':
    main()
