"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE'S OWN SOURCE (progen_transformer/{progen,utils}.py of a
lucidrains/progen checkout, unmodified) under the numpy stand-ins in oracle/ref_shim/ (jax/haiku are not installable).
The tests only read the stored files; regenerating needs the checkout:
    python tests/golden/make_golden.py PATH_TO_LUCIDRAINS_PROGEN

For each case the parameters come from the oracle's seeded initialiser (`init_params` + `randomize_params`,
numpy default_rng => reproducible), are fed to the reference `model.apply`, and the reference's logits, loss
(`utils.cross_entropy`) and greedy samples (`utils.sample` with zero gumbel noise) are stored.  Gradient
fingerprints come from the torch twin (the reference's `value_and_grad` needs real jax) and are marked as such.
"""
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

CASES = {
    # name: (constructor kwargs, param seed, data seed)
    'tiny_glu_sgu': (dict(num_tokens=256, dim=64, seq_len=32, depth=3, window_size=8, global_mlp_depth=1,
                          heads=2, dim_head=32), 11, 12),
    'tiny_gelu_sgu': (dict(num_tokens=256, dim=64, seq_len=64, depth=2, window_size=16, global_mlp_depth=1,
                           heads=4, dim_head=16, ff_glu=False), 21, 22),
    'tiny_all_glu': (dict(num_tokens=256, dim=128, seq_len=128, depth=2, window_size=64, global_mlp_depth=0,
                          heads=2, dim_head=64), 31, 32),
    # BASELINE.json configs[0]: dim=512 depth=2 seq_len=1024 window=256 (constructor defaults otherwise, so
    # global_mlp_depth=2 makes BOTH layers gMLP/SGU layers)
    'cfg1': (dict(num_tokens=256, dim=512, seq_len=1024, depth=2, window_size=256), 41, 42),
}
CFG1_ROWS = np.arange(0, 1024, 16)       # logits rows kept for cfg1 (64 x 256)


def fingerprint(params):
    return float(sum(np.abs(a.astype(np.float64)).sum() for d in params.values() for a in d.values()))


def make_inputs(kwargs, pseed, dseed, B=2):
    from oracle import progen_ref as O
    cfg = O.make_config(**kwargs)
    params = O.randomize_params(O.init_params(cfg, pseed), pseed + 1000)
    rng = np.random.default_rng(dseed)
    data = rng.integers(0, 256, (B, cfg['seq_len'] + 1)).astype(np.uint16)
    # one row with an early end-of-string followed by padding, to exercise the loss mask (utils.py:54-56)
    data[1, cfg['seq_len'] // 2:] = 0
    return cfg, params, data


def main(reference_dir):
    from oracle import progen_ref as O
    from oracle import progen_torch as T
    inputs = {name: make_inputs(*spec) for name, spec in CASES.items()}

    # ---- reference source under the shim
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'ref_shim'))
    sys.path.insert(0, reference_dir)
    import haiku as hk
    from progen_transformer.progen import ProGen
    from progen_transformer import utils as RU

    for name, (kwargs, pseed, dseed) in CASES.items():
        cfg, params, data = inputs[name]
        model = ProGen(**kwargs)
        # the reference's own init gives the parameter tree structure (module paths + shapes) to check ours
        ref_tree = model.init(np.array([0, 1]), np.zeros(cfg['seq_len'], np.int64))
        assert {m: {k: v.shape for k, v in d.items()} for m, d in ref_tree.items()} == \
               {m: {k: v.shape for k, v in d.items()} for m, d in params.items()}, 'param tree mismatch'
        p64 = {m: {k: v.astype(np.float64) for k, v in d.items()} for m, d in params.items()}
        logits = np.stack([np.asarray(model.apply(p64, None, row[:-1].astype(np.int64))) for row in data])
        ce = np.stack([np.asarray(RU.cross_entropy(logits[b], data[b, 1:].astype(np.int64))) for b in range(len(data))])
        out = dict(param_seed=pseed, data_seed=dseed, param_fingerprint=fingerprint(params),
                   data=data, ce_per_row=ce, loss=ce.mean())
        if name == 'cfg1':
            out['logits_rows'] = CFG1_ROWS
            out['logits'] = logits[:, CFG1_ROWS].astype(np.float32)
            out['logits_absmax'] = np.abs(logits).max()
        else:
            out['logits'] = logits
            # greedy samples from the reference sampler (zero noise): with and without add_bos, top_k=25
            prime = data[0, 1:6].astype(np.uint16)
            for add_bos in (False, True):
                s = RU.sample(hk.PRNGSequence(0), model.apply, p64, prime.copy(), cfg['seq_len'], top_k=25,
                              add_bos=add_bos)
                out[f'sample_bos{int(add_bos)}'] = np.asarray(s).astype(np.int64)
            out['prime'] = prime
            # gradient fingerprints (torch twin, NOT the reference's value_and_grad)
            loss_t, grads = T.loss_and_grads(params, data, cfg)
            assert abs(loss_t - float(ce.mean())) < 1e-10, (loss_t, ce.mean())
            keys = sorted((m, k) for m, d in grads.items() for k in d)
            out['grad_keys'] = np.array([f'{m}|{k}' for m, k in keys])
            out['grad_norms'] = np.array([np.linalg.norm(grads[m][k]) for m, k in keys])
            out['grad_head'] = np.stack([np.resize(grads[m][k].ravel()[:8], 8) for m, k in keys])
        path = os.path.join(ROOT, 'tests', 'golden', f'{name}.npz')
        np.savez_compressed(path, **out)
        print(name, 'loss', float(ce.mean()), 'logits absmax', float(np.abs(logits).max()),
              os.path.getsize(path) // 1024, 'KiB')


if __name__ == '__main__':
    if len(sys.argv) != 2:
        sys.exit('usage: python tests/golden/make_golden.py PATH_TO_LUCIDRAINS_PROGEN')
    main(sys.argv[1])
