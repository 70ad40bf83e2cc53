"""Host side of `train_mode=scst` (stays Python, as in the reference).

  id_to_caption              src/infer_fn.py:36-75
  radix_wtoi / captions_to_batched_ids
                             common/inputs/manager_image_caption.py:240-254, 477-509
  CaptionScorer              common/scst/scorers.py:30-197  (weighted CIDEr-D + BLEU reward,
                             greedy baseline tiled over the beam)
  CiderD                     common/scst/cider_ruotianluo/pyciderevalcap/ciderD/ciderD_scorer.py
                             (tf-idf n-gram cosine with clipping and the gaussian length
                             penalty; cached document frequencies)
  bleu_closest               common/coco_caption/pycocoevalcap/bleu/bleu_scorer.py:23-83,198-263
                             (per-sentence BLEU-1..4, `closest` reference length) -- the
                             reference file is Python-2-only syntax, so it is restated here
  compute_doc_freq           common/scst/prepro_ngrams.py:61-73
  scst_step                  src/train_fn.py:218-256 (sample -> host reward -> weighted XE)

The n-gram statistics are plain dict / Counter work on a few hundred short sentences
per step; the GPU does the sampling (greedy + beam search) and the training step.
"""
from __future__ import annotations

import functools
import math
import pickle
from collections import Counter, defaultdict

import numpy as np

from .engine import executed_steps
from .model import number_to_base


# ---------------------------------------------------------------------------
# ids <-> captions
# ---------------------------------------------------------------------------
def id_to_caption(ids, config):
    """src/infer_fn.py:46-75.  ids [N, T] int."""
    c = config
    ids = np.asarray(ids)
    captions = []
    if c.token_type == 'radix':
        base = c.radix_base
        vocab_size = len(c.itow)
        word_len = len(number_to_base(vocab_size, base))
        for i in range(ids.shape[0]):
            row = [int(w) for w in ids[i, :] if 0 <= w < base]
            if len(row) % word_len != 0:
                row = row[:-1]
            sent = []
            for j in range(0, len(row), word_len):
                word_id = 0
                for d in row[j:j + word_len]:
                    word_id = word_id * base + d
                if word_id < vocab_size:
                    sent.append(c.itow[str(word_id)])
            captions.append(' '.join(sent))
    else:
        eos = c.wtoi['<EOS>']
        joiner = ' ' if c.token_type == 'word' else ''
        for i in range(ids.shape[0]):
            row = [int(w) for w in ids[i, :] if w >= 0 and w != eos]
            # (JSON-loaded tables are str-keyed; the char table InputManager_Char builds is int-keyed and leaves id 37
            # unassigned -- the reference would raise KeyError on it; it is skipped here)
            toks = [c.itow.get(str(w), c.itow.get(w)) for w in row]
            captions.append(joiner.join(t for t in toks if t is not None))
    return captions


def build_radix_wtoi(config):
    """common/inputs/manager_image_caption.py:240-254."""
    c = config
    max_word_len = len(number_to_base(len(c.wtoi), c.radix_base))
    assert c.wtoi['<PAD>'] == -1
    out = {}
    for k, v in c.wtoi.items():
        if k == '<GO>':
            idx = [c.radix_base]
        elif k == '<EOS>':
            idx = [c.radix_base + 1]
        elif k == '<PAD>':
            idx = [-1]
        else:
            idx = number_to_base(v, c.radix_base)
            idx = [0] * (max_word_len - len(idx)) + idx
        out[k] = idx
    return out


_RADIX_TABLES = {}       # id(wtoi) -> (wtoi, radix_base, table)


def captions_to_batched_ids(hypos, config, radix_wtoi=None):
    """common/inputs/manager_image_caption.py:477-509.  hypos: list of [caption string]."""
    c = config
    assert c.token_type in ['radix', 'word', 'char']
    rows = []
    if c.token_type == 'radix' and radix_wtoi is None:
        # the table is a function of the vocabulary alone (the reference's InputManager_Radix builds it once in __init__):
        # cached per vocabulary object -- rebuilding it cost 15 ms of every 32 ms SCST step (profiles/r09f_scst_profile.txt)
        cache = _RADIX_TABLES.get(id(c.wtoi))
        if cache is None or cache[0] is not c.wtoi or cache[1] != c.radix_base:
            cache = _RADIX_TABLES[id(c.wtoi)] = (c.wtoi, c.radix_base, build_radix_wtoi(c))
        radix_wtoi = cache[2]
    for h in hypos:
        if c.token_type == 'radix':
            toks = ['<GO>'] + h[0].split() + ['<EOS>']
            ids = [d for w in toks for d in radix_wtoi.get(w, radix_wtoi['<UNK>'])]
        elif c.token_type == 'word':
            toks = ['<GO>'] + h[0].split() + ['<EOS>']
            ids = [c.wtoi.get(w, c.wtoi['<UNK>']) for w in toks]
        else:
            ids = [c.wtoi['<GO>']] + [c.wtoi[ch] for ch in h[0]] + [c.wtoi['<EOS>']]
        rows.append(ids)
    max_len = max(len(r) for r in rows)
    assert max_len > 1
    out = np.full((len(rows), max_len), c.wtoi['<PAD>'], np.int32)
    for i, r in enumerate(rows):
        out[i, :len(r)] = r
    return out


# ---------------------------------------------------------------------------
# n-gram statistics
# ---------------------------------------------------------------------------
@functools.lru_cache(maxsize=65536)
def ngram_counts(sentence, n=4):
    """`precook`: Counter of all 1..n-grams (as tuples) of a whitespace-tokenised string.  Memoised (the
    result is treated as read-only): CIDEr-D and BLEU cook the same hypothesis, and the training set's
    reference captions come back every epoch."""
    words = sentence.split()
    counts = Counter()
    for k in range(1, n + 1):
        for i in range(len(words) - k + 1):
            counts[tuple(words[i:i + k])] += 1
    return len(words), counts


def compute_doc_freq(refs_per_image, n=4):
    """common/scst/prepro_ngrams.py:61-73: in how many images does an n-gram occur."""
    df = defaultdict(float)
    for refs in refs_per_image:
        seen = set()
        for r in refs:
            seen.update(ngram_counts(r, n)[1].keys())
        for g in seen:
            df[g] += 1
    return df


class CiderD(object):
    """CIDEr-D with cached document frequencies (ciderD_scorer.py:52-222).
    `df`: path to a pickle {document_frequency, ref_len}, such a dict, or 'corpus'."""

    def __init__(self, n=4, sigma=6.0, df='corpus'):
        self.n, self.sigma = n, sigma
        self.df_mode = df
        self.document_frequency = None
        self.ref_len = None
        if isinstance(df, dict):
            self.document_frequency = df['document_frequency']
            self.ref_len = math.log(float(df['ref_len']))
        elif df != 'corpus':
            with open(df, 'rb') as f:
                try:
                    p = pickle.load(f)
                except UnicodeDecodeError:
                    f.seek(0)
                    p = pickle.load(f, encoding='latin1')
            self.document_frequency = p['document_frequency']
            self.ref_len = math.log(float(p['ref_len']))

    def _vec(self, counts, dfreq, ref_len):
        vec = [dict() for _ in range(self.n)]
        norm = [0.0] * self.n
        length = 0
        for ngram, tf in counts.items():
            d = math.log(max(1.0, dfreq.get(ngram, 0.0)))
            k = len(ngram) - 1
            w = float(tf) * (ref_len - d)
            vec[k][ngram] = w
            norm[k] += w * w
            if k == 1:                      # the reference counts bigrams here (ciderD_scorer.py:152)
                length += tf
        return vec, [math.sqrt(x) for x in norm], length

    def compute_score(self, gts, res):
        """gts: {id: [ref strings]}, res: {id: [hypothesis string]} -> (mean, scores in id order of gts)."""
        assert sorted(gts.keys()) == sorted(res.keys())
        ids = list(gts.keys())
        # the SCST loop scores k sampled captions + 1 greedy caption per image against the SAME reference list
        # object (CaptionScorer.get_hypo_scores): cook / weight each distinct list once (same arithmetic)
        cooked = {}
        for i in ids:
            if id(gts[i]) not in cooked:
                cooked[id(gts[i])] = [ngram_counts(r, self.n)[1] for r in gts[i]]
        crefs = [cooked[id(gts[i])] for i in ids]
        ctest = [ngram_counts(res[i][0], self.n)[1] for i in ids]
        if self.df_mode == 'corpus' and not isinstance(self.df_mode, dict):
            dfreq = defaultdict(float)
            for refs in crefs:
                for g in set(g for r in refs for g in r):
                    dfreq[g] += 1
            ref_len = math.log(float(len(crefs)))
        else:
            dfreq, ref_len = self.document_frequency, self.ref_len
        scores = []
        ref_vecs = {}
        for test, refs in zip(ctest, crefs):
            vec, norm, length = self._vec(test, dfreq, ref_len)
            score = np.zeros(self.n)
            if id(refs) not in ref_vecs:
                ref_vecs[id(refs)] = [self._vec(ref, dfreq, ref_len) for ref in refs]
            for vr, nr, lr in ref_vecs[id(refs)]:
                delta = float(length - lr)
                pen = math.e ** (-(delta ** 2) / (2 * self.sigma ** 2))
                for k in range(self.n):
                    v = 0.0
                    rk = vr[k]
                    for g, w in vec[k].items():
                        wr = rk.get(g)
                        if wr is None:
                            continue            # min(w, 0.0) * 0.0 adds a (signed) zero: v is unchanged
                        v += min(w, wr) * wr
                    if norm[k] != 0 and nr[k] != 0:
                        v /= (norm[k] * nr[k])
                    score[k] += v * pen
            scores.append(float(np.mean(score)) / len(refs) * 10.0)
        scores = np.array(scores)
        return float(scores.mean()), scores


def bleu_closest(gts, res, n=4):
    """BleuScorer.compute_score(option='closest') (bleu_scorer.py:198-263) through
    BleuSilent (scorers.py:174-197): returns (corpus BLEU-1..n, per-sentence lists [n][N])."""
    small, tiny = 1e-9, 1e-15
    bleu_list = [[] for _ in range(n)]
    tot_test, tot_ref = 0, 0
    tot_guess, tot_correct = [0] * n, [0] * n
    ref_stats = {}                                      # per distinct reference list (see CiderD.compute_score)
    for i in gts:
        hypo, refs = res[i], gts[i]
        assert isinstance(hypo, list) and len(hypo) == 1 and isinstance(refs, list) and len(refs) >= 1
        if id(refs) not in ref_stats:
            reflens, maxcounts = [], {}
            for r in refs:
                rl, cnt = ngram_counts(r, n)
                reflens.append(rl)
                for g, ct in cnt.items():
                    if ct > maxcounts.get(g, 0):
                        maxcounts[g] = ct
            ref_stats[id(refs)] = (reflens, maxcounts)
        reflens, maxcounts = ref_stats[id(refs)]
        testlen, counts = ngram_counts(hypo[0], n)
        reflen = min((abs(l - testlen), l) for l in reflens)[1]
        guess = [max(0, testlen - k + 1) for k in range(1, n + 1)]
        correct = [0] * n
        for g, ct in counts.items():
            correct[len(g) - 1] += min(maxcounts.get(g, 0), ct)
        tot_test += testlen
        tot_ref += reflen
        b = 1.0
        for k in range(n):
            tot_guess[k] += guess[k]
            tot_correct[k] += correct[k]
            b *= (float(correct[k]) + tiny) / (float(guess[k]) + small)
            bleu_list[k].append(b ** (1.0 / (k + 1)))
        ratio = (testlen + tiny) / (reflen + small)
        if ratio < 1:
            for k in range(n):
                bleu_list[k][-1] *= math.exp(1 - 1 / ratio)
    bleus = []
    b = 1.0
    for k in range(n):
        b *= float(tot_correct[k] + tiny) / (tot_guess[k] + small)
        bleus.append(b ** (1.0 / (k + 1)))
    ratio = (tot_test + tiny) / (tot_ref + small)
    if ratio < 1:
        bleus = [x * math.exp(1 - 1 / ratio) for x in bleus]
    return bleus, bleu_list


class CaptionScorer(object):
    """common/scst/scorers.py:30-171 (`captionScorer`)."""

    def __init__(self, path_to_cached_tokens, metric_weights):
        # the reference also offers plain 'cider' (common/scst/scorers.py:36-39); it is not built here, and a
        # positive weight on a metric that contributes nothing would silently change the reward
        for key, wt in dict(metric_weights).items():
            if key not in ('ciderD', 'bleu') and np.amax(np.asarray(wt, np.float64)) > 0:
                raise NotImplementedError("metric '%s' is not built (ciderD and bleu are)" % key)
        self._ciderD = CiderD(df=path_to_cached_tokens)
        self.weights = metric_weights

    def get_hypo_scores(self, refs, sample, greedy, best_hypo_only=False):
        assert isinstance(refs, list) and isinstance(sample, list) and isinstance(greedy, list)
        assert isinstance(refs[0], list) and isinstance(sample[0], list) and isinstance(greedy[0], list)
        assert len(refs) == len(greedy)
        assert len(sample) % len(greedy) == 0
        num_sample, num_greedy = len(sample), len(greedy)
        multiple = num_sample // num_greedy
        gts, res = {}, {}
        for idx in range(num_sample):                       # key order [greedy, sampled]
            if idx < num_greedy:
                res[idx] = greedy[idx]
                gts[idx] = refs[idx]
            res[idx + num_greedy] = sample[idx]
            gts[idx + num_greedy] = refs[idx % num_greedy]
        keys = sorted(gts.keys())
        gts = {k: gts[k] for k in keys}
        res = {k: res[k] for k in keys}
        total = np.zeros(num_sample + num_greedy)
        w = self.weights
        if 'ciderD' in w and np.amax(w['ciderD']) > 0:
            total = total + self._ciderD.compute_score(gts, res)[1] * w['ciderD']
        if 'bleu' in w and np.amax(w['bleu']) > 0:
            _, per = bleu_closest(gts, res, 4)
            for i, wi in enumerate(w['bleu']):
                total = total + np.array(per[i]) * wi
        sc_greedy = total[:num_greedy]
        sc_sample = total[num_greedy:]
        if num_sample > num_greedy and best_hypo_only:
            sc = np.reshape(sc_sample, [multiple, num_greedy])
            best = np.argmax(sc, axis=0)
            final_hypo = [sample[idx + num_greedy * best[idx]] for idx in range(num_greedy)]
            sc_sample = np.amax(sc, axis=0)
        else:
            if num_sample > num_greedy:
                sc_greedy = np.concatenate([sc_greedy] * multiple)
            final_hypo = sample
        return final_hypo, sc_sample, sc_greedy


# ---------------------------------------------------------------------------
# One SCST step (src/train_fn.py:218-256)
# ---------------------------------------------------------------------------
def sample_captions(engine, config, images, beam, max_length=20):
    """CaptionModel_SCST('sample') (src/model.py:121-126, model_base.py:203-215): greedy decode
    + beam-`beam` search, infer_max_length 20, length penalty 0, no dropout.  The encoder and
    the key projection run ONCE per image for both decodes.  Returns (cap_beam [k,B,T] int32,
    cap_greedy [B,T] int32, im_embed, fm)."""
    c = config
    max_it = max_length
    if c.token_type == 'radix':
        max_it *= len(number_to_base(len(c.wtoi), c.radix_base))
    elif c.token_type == 'char':
        max_it *= 5
    im_embed, fm = engine.encode(images)
    keys, values = engine.project_fm(fm)
    c0, h0 = engine.rnn_init(im_embed)
    g = engine.decode_greedy(keys, values, c0, h0, max_it, want_logits=False, want_attn=False)
    b = engine.decode_beam(keys, values, c0, h0, beam, 0.0, max_it, want_attn=False)
    Tg, Tb = executed_steps(g['T']), executed_steps(b['T'])
    cap_greedy = g['ids'][:Tg].transpose(0, 1).contiguous()              # [B, T]
    cap_beam = b['predicted_ids'][:Tb].permute(2, 1, 0).contiguous()     # [k, B, T]  (top_beam=False, :286-288)
    return cap_beam, cap_greedy, im_embed, fm


def scst_step(trainer, scorer, images, refs, seed=None, lr=None, dropout=True):
    """train_fn_scst loop body.  images [B,224,224,3] fp32 device tensor, or raw uint8 pixels (a [B,H,W,3] tensor or a
    list of [h,w,3] arrays of mixed sizes) pre-processed on the device as `Trainer.prepare_images` does; refs: list (per
    image) of reference caption strings.  Returns dict(loss, rewards, sc_sample, sc_greedy, hypos) plus the
    augmentation draws crop_yx / flip of raw pixels under `cnn_input_augment`."""
    c, eng = trainer.c, trainer.engine
    k = c.scst_beam_size
    images, draws = trainer.prepare_images(images, seed)
    cap_beam, cap_greedy, im_embed, fm = sample_captions(eng, c, images, k)
    cb = cap_beam.cpu().numpy()
    cb = cb.reshape(-1, cb.shape[-1])                                     # [[im0_h0]..[imN_h0],[im0_h1]..]
    hyp_beam = [[s] for s in id_to_caption(cb, c)]
    hyp_greedy = [[s] for s in id_to_caption(cap_greedy.cpu().numpy(), c)]
    hypos, sc_sample, sc_greedy = scorer.get_hypo_scores(refs, hyp_beam, hyp_greedy)
    rewards = (sc_sample - sc_greedy).astype(np.float32)
    hypos_idx = captions_to_batched_ids(hypos, c)
    assert hypos_idx.shape[0] == sc_sample.shape[0]
    # the reference re-encodes the k-times tiled images (train_fn.py:251); the CNN is frozen and
    # deterministic, so the encoder outputs are repeated instead
    fm_t = fm.repeat(k, 1, 1)
    im_t = im_embed.repeat(k, 1)
    masks, keeps = None, (1.0, 1.0, 1.0)
    if dropout:
        from .train import process_inputs
        lens = process_inputs(hypos_idx, c.token_type)[3]
        masks, keeps = trainer.make_masks(fm_t.shape[0], int(lens.max()), trainer.dropout_seed(seed))
    out = trainer.forward_backward(fm_t, im_t, hypos_idx, rewards, masks, keeps)
    out['lr'] = trainer.apply_gradients(lr)
    out.update(rewards=rewards, sc_sample=sc_sample, sc_greedy=sc_greedy, hypos=hypos, greedy=hyp_greedy)
    if draws:
        out.update(draws)
    return out
