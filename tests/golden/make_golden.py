"""Generates the committed golden fixtures in this directory from the NumPy oracle.

    python tests/golden/make_golden.py [REFERENCE_CHECKOUT]    # rewrites *.npz (and the reference's records)

The reference itself (TF 1.9 / Python 2.7) cannot run under Python 3, so the
fixtures are outputs of `oracle/` on seeded inputs, not of the reference; they
freeze the oracle (tests/test_oracle_known_answers.py) and give the CUDA path a
target that does not move (tests/test_gpu_parity.py::test_golden_*).  Two
records come from a checkout of the reference and are rewritten only when one
is given:
- ciderd_reference.npz: outputs of the reference's CIDEr-D scorer
  (common/scst/cider_ruotianluo/pyciderevalcap/ciderD, the one piece of it that
  imports under Python 3) for the SCST reward;
- reference_cli_flags.json: name, type, default and choices of every flag of
  the reference's src/train.py and src/infer.py parsers.  The committed table
  was written from comic_b200.cli's parsers after they had been matched flag by
  flag against those sources by `reference_cli_flags()`.
"""
import ast
import json
import os
import re
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (ROOT, os.path.join(ROOT, 'oracle'), os.path.join(ROOT, 'tests')):
    if p not in sys.path:
        sys.path.insert(0, p)

import comic_b200  # noqa: E402,F401
from comic_b200 import configuration as conf  # noqa: E402
from comic_b200 import weights as wts  # noqa: E402
import comic_oracle as O  # noqa: E402
import inception_v1_oracle as I  # noqa: E402


def golden_weights(c, include_cnn):
    return wts.perturb_for_parity(wts.init_weights(c, seed=20240101, cnn_init='he', include_cnn=include_cnn))


def decoder_inputs(B, seed):
    rng = np.random.default_rng(seed)
    fm = np.maximum(rng.standard_normal((B, 196, 832)), 0).astype(np.float32)
    im = np.maximum(rng.standard_normal((B, 1024)), 0).astype(np.float32)
    return im, fm


def decoder_beam_case():
    """COMIC-256 beam-3, 4 images, 10 radix steps."""
    c = conf.make_config()
    W = golden_weights(c, False)
    im, fm = decoder_inputs(4, 77)
    r = O.beam_search_decode(O.Decoder(W, c), im, fm, 3, 0.0, 10)
    _, _, am = O.post_process_beam(r, 8, 3)
    return dict(predicted_ids=r['predicted_ids'], parent_ids=r['parent_ids'], step_ids=r['step_ids'],
                lengths=r['lengths'], scores=r['scores'], attn_top=am.astype(np.float32))


def encoder_case():
    """2 images through InceptionV1: im_embed, a strided sample of Mixed_4f and its sum."""
    c = conf.make_config()
    W = golden_weights(c, True)
    rng = np.random.default_rng(5)
    img = rng.uniform(-1, 1, (2, 224, 224, 3)).astype(np.float32)
    emb, fm, _ = I.encoder(img, W, c)
    return dict(im_embed=emb, fm_sample=fm[:, ::7, ::13].copy(), fm_sum=np.float64(fm.astype(np.float64).sum()))


def scst_sentences(seed=11, n_img=6, n_ref=5, n_hyp=3, vocab=40):
    """Random short sentences over a small vocabulary (so n-grams overlap)."""
    rng = np.random.default_rng(seed)
    mk = lambda: ' '.join('w%d' % w for w in rng.integers(0, vocab, size=int(rng.integers(3, 12))))
    refs = [[mk() for _ in range(n_ref)] for _ in range(n_img)]
    hyps = []
    for i in range(n_img):
        for j in range(n_hyp):
            base = refs[i][j % n_ref].split()
            keep = [w for w in base if rng.uniform() < 0.7] or base[:1]
            hyps.append(' '.join(keep + ['w%d' % rng.integers(0, vocab)]))
    hyps.append('')                                           # empty hypothesis edge case
    return refs, hyps


def ciderd_case(reference):
    """CIDEr-D scores from the REFERENCE's own scorer (the one module of the reference checkout that
    imports under Python 3), cached-DF mode (the mode train_fn_scst uses)."""
    import pickle
    import tempfile
    sys.path.insert(0, os.path.join(reference, 'common', 'scst', 'cider_ruotianluo'))
    from pyciderevalcap.ciderD.ciderD import CiderD as RefCiderD
    from comic_b200 import scst as S
    refs, hyps = scst_sentences()
    n_img = len(refs)
    gts = {i: refs[i % n_img] for i in range(len(hyps))}
    res = {i: [hyps[i]] for i in range(len(hyps))}
    df = S.compute_doc_freq(refs)
    with tempfile.NamedTemporaryFile(suffix='.p', delete=False) as f:
        pickle.dump({'document_frequency': df, 'ref_len': n_img}, f, 2)
        path = f.name
    mean_c, sc_c = RefCiderD(df=path).compute_score(gts, res)     # (df='corpus' raises in the reference: copy_empty)
    os.unlink(path)
    return dict(cached=np.asarray(sc_c, np.float64), mean_cached=np.float64(mean_c))


PATH_FLAGS = ('infer_checkpoints_dir', 'dataset_dir')      # defaults are path expressions of the reference's checkout


def reference_cli_flags(reference):
    """{'train.py' | 'infer.py': {flag: {'type', 'default', 'choices'}}} parsed from the add_argument calls of the
    reference's src/train.py and src/infer.py (no default recorded for PATH_FLAGS)."""
    out = {}
    for fname in ('train.py', 'infer.py'):
        with open(os.path.join(reference, 'src', fname)) as f:
            src = f.read()
        flags = {}
        for m in re.finditer(r"add_argument\(\s*'--(\w+)'(.*?)help=", src, re.S):
            name, body = m.group(1), m.group(2)
            t = re.search(r"type=(\w+)", body)
            d = re.search(r"default=(.+?),\s*(?:choices=|$)", body.strip(), re.S)
            c = re.search(r"choices=(\[.*?\])", body, re.S)
            spec = {'type': t.group(1) if t else None}
            if name not in PATH_FLAGS:
                spec['default'] = eval(d.group(1).strip().rstrip(',')) if d else None
            spec['choices'] = ast.literal_eval(c.group(1)) if c else None
            flags[name] = spec
        out[fname] = flags
    return out


def write_reference_cli_flags(table, path):
    """One line per flag, so that a change of the table reads as a change of that flag."""
    lines = []
    for fname, flags in table.items():
        rows = ['  %s: %s' % (json.dumps(name), json.dumps(spec)) for name, spec in flags.items()]
        lines.append(' %s: {\n%s\n }' % (json.dumps(fname), ',\n'.join(rows)))
    with open(path, 'w') as f:
        f.write('{\n%s\n}\n' % ',\n'.join(lines))


def main(argv):
    np.savez_compressed(os.path.join(HERE, 'decoder_beam_comic256.npz'), **decoder_beam_case())
    np.savez_compressed(os.path.join(HERE, 'encoder_2img.npz'), **encoder_case())
    if argv:
        reference = argv[0]
        np.savez_compressed(os.path.join(HERE, 'ciderd_reference.npz'), **ciderd_case(reference))
        write_reference_cli_flags(reference_cli_flags(reference), os.path.join(HERE, 'reference_cli_flags.json'))
    print('wrote fixtures to', HERE)


if __name__ == '__main__':
    main(sys.argv[1:])
