"""Generate golden fixtures by running the UNMODIFIED reference.

    python tests/golden/make_golden.py [fixture ...]      (default: all of them)

The reference is read from oracle/_ref (a git-ignored checkout of the upstream
project) or from the directory SCONE_REFERENCE_ROOT names.

Imports ``NGramExtractor`` / ``EmbeddingCache`` from that checkout through
``oracle/ref_shim.py`` and records their outputs on seeded inputs into small
``.npz`` files next to this script.  The reference is not part of this
repository, so the tests read only the committed ``.npz`` files.

What each fixture pins (reference file:line):
  kat0.npz        fit + longest match on the hand-sized case of SURVEY.md 8c
                  (n_gram_extractor.py:72-104, :106-126; embedding_cache.py:173)
  fit_small.npz   fit (truncate-then-filter, tie order) on a seeded Zipf corpus,
                  longest match on a [B, L] batch incl. rows crossing nothing,
                  and the raw all-containing lists of get_token_f_grams
  fit_medium.npz  fit on 300 texts / 60 k tokens with max_f_grams = 3000: the cut falls
                  inside a run of equal counts (first-seen order decides), texts
                  shorter than max_n (n_gram_extractor.py:58-70, :91-99)
  vocab_n5.npz    a max_n = 5 vocabulary WITHOUT unigrams (lengths 2..5, set
                  directly on the extractor the way NGramExtractor.load does,
                  n_gram_extractor.py:159-165), longest match on a batch
  cache_small.npz EmbeddingCache.cache_embeddings / get_embeddings (dict and
                  memmap backends, embedding_cache.py:56-147), `.half()` of the
                  gathered rows (engine.py:265-266), and the engine's assemble
                  loop (engine.py:235-259) re-enacted on the reference objects
  live_2024.npz   fit (max_n = 4, min_freq = 2, max_f_grams = 500) on a 30-text Zipf(1.2)
                  corpus over 60 tokens and get_token_f_grams of a 120-token query
                  (tests/test_oracle.py::test_live_reference_agrees_with_oracle)
"""

from __future__ import annotations

import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))

from oracle import ref_shim  # noqa: E402

NGramExtractor, EmbeddingCache = ref_shim.load_reference()


def vocab_arrays(ex, max_n):
    N = len(ex.id_to_f_gram)
    toks = np.full((N, max_n), -1, dtype=np.int32)
    lens = np.zeros(N, dtype=np.uint8)
    for i in range(N):
        g = ex.id_to_f_gram[i]
        toks[i, :len(g)] = g
        lens[i] = len(g)
    return toks, lens


def ref_longest(ex, row):
    """SURVEY.md 0.4: the reference primitive applied to each max_n window."""
    L = len(row)
    ids = np.full(L, -1, dtype=np.int32)
    lens = np.zeros(L, dtype=np.uint8)
    for i in range(L):
        lo = max(0, i - ex.max_n + 1)
        w = row[lo:i + 1]
        hits = ex.get_token_f_grams(w)[len(w) - 1]
        if hits:
            ids[i] = ex.f_gram_to_id[hits[-1]]
            lens[i] = len(hits[-1])
    return ids, lens


def ref_longest_batch(ex, ids2d):
    out_i = np.zeros(ids2d.shape, dtype=np.int32)
    out_l = np.zeros(ids2d.shape, dtype=np.uint8)
    for b in range(ids2d.shape[0]):
        out_i[b], out_l[b] = ref_longest(ex, [int(t) for t in ids2d[b]])
    return out_i, out_l


def ref_containing(ex, row):
    """Flatten get_token_f_grams(row) -> (offsets [L+1], gram ids in list order)."""
    tf = ex.get_token_f_grams(row)
    offs, flat = [0], []
    for pos in range(len(row)):
        flat.extend(ex.f_gram_to_id[g] for g in tf[pos])
        offs.append(len(flat))
    return np.array(offs, dtype=np.int32), np.array(flat, dtype=np.int32)


def zipf_tokens(rng, n, V, a=1.2):
    return (rng.zipf(a, size=n) - 1) % V


def make_kat0():
    ex = NGramExtractor(max_n=3, min_freq=1, max_f_grams=100).fit([[1, 2, 3, 4, 1, 2, 3], [2, 3, 4, 5], [1, 2, 9]], verbose=False)
    toks, lens = vocab_arrays(ex, 3)
    q = [1, 2, 3, 7, 1, 2, 3, 4, 5, 9, 2, 3]
    ids, ml = ref_longest(ex, q)
    ex2 = NGramExtractor(max_n=2, min_freq=2, max_f_grams=3).fit([[7, 8, 7, 8, 9]], verbose=False)
    t2, l2 = vocab_arrays(ex2, 2)
    np.savez_compressed(os.path.join(HERE, "kat0.npz"), vocab_tokens=toks, vocab_lens=lens,
                        query=np.array(q, dtype=np.int64), fgram_id=ids, match_len=ml,
                        vocab2_tokens=t2, vocab2_lens=l2)


def make_fit_small():
    rng = np.random.default_rng(1234)
    V = 400
    corpus = [zipf_tokens(rng, int(rng.integers(5, 61)), V, a=1.1).tolist() for _ in range(40)]
    max_n, min_freq, max_f = 3, 2, 400
    ex = NGramExtractor(max_n=max_n, min_freq=min_freq, max_f_grams=max_f).fit(corpus, verbose=False)
    toks, lens = vocab_arrays(ex, max_n)
    B, L = 6, 48
    q = zipf_tokens(rng, B * L, V, a=1.1).reshape(B, L).astype(np.int64)
    q[2, :] = 0            # a row of pads: pads are ordinary tokens (f_gram_tokenizer.py:122-123)
    q[3, 10:20] = 399      # a rare token run
    q[4, :5] = corpus[0][:5]
    fid, ml = ref_longest_batch(ex, q)
    offs, flat = zip(*[ref_containing(ex, [int(t) for t in q[b]]) for b in range(B)])
    corpus_flat = np.concatenate([np.array(c, dtype=np.int64) for c in corpus])
    corpus_offs = np.cumsum([0] + [len(c) for c in corpus]).astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "fit_small.npz"), corpus_flat=corpus_flat, corpus_offs=corpus_offs,
                        max_n=max_n, min_freq=min_freq, max_f_grams=max_f,
                        vocab_tokens=toks, vocab_lens=lens, query=q, fgram_id=fid, match_len=ml,
                        cont_offs=np.stack(offs), cont_flat=np.concatenate(flat),
                        cont_flat_offs=np.cumsum([0] + [len(f) for f in flat]).astype(np.int64))


def make_fit_medium():
    """A corpus large enough for the things fit_small cannot show: thousands of n-grams TIED at the truncation boundary (the
    reference keeps first-seen order among equal counts: Counter.most_common is a stable sort) and texts shorter than max_n."""
    rng = np.random.default_rng(4321)
    V = 2000
    lens_ = [int(x) for x in rng.integers(1, 400, size=300)]
    lens_[7], lens_[8], lens_[9] = 1, 2, 3                      # shorter than max_n
    corpus = [zipf_tokens(rng, n, V, a=1.05).tolist() for n in lens_]
    max_n, min_freq, max_f = 4, 3, 3000
    ex = NGramExtractor(max_n=max_n, min_freq=min_freq, max_f_grams=max_f).fit(corpus, verbose=False)
    toks, lens = vocab_arrays(ex, max_n)
    corpus_flat = np.concatenate([np.array(c, dtype=np.int32) for c in corpus])
    corpus_offs = np.cumsum([0] + [len(c) for c in corpus]).astype(np.int64)
    np.savez_compressed(os.path.join(HERE, "fit_medium.npz"), corpus_flat=corpus_flat, corpus_offs=corpus_offs,
                        max_n=max_n, min_freq=min_freq, max_f_grams=max_f, vocab_tokens=toks, vocab_lens=lens)
    return ex


def make_vocab_n5():
    rng = np.random.default_rng(77)
    V, max_n, N = 300, 5, 1500
    grams, seen = [], set()
    # nested families so that shorter suffixes of longer f-grams are present too
    while len(grams) < N:
        n = int(rng.integers(2, max_n + 1))
        g = tuple(int(t) for t in zipf_tokens(rng, n, V, a=1.15))
        for k in (n, max(2, n - 1)):
            s = g[n - k:]
            if s not in seen and len(grams) < N:
                seen.add(s)
                grams.append(s)
    ex = NGramExtractor(max_n=max_n, min_freq=1, max_f_grams=N)
    ex.f_gram_to_id = {g: i for i, g in enumerate(grams)}
    ex.id_to_f_gram = {i: g for i, g in enumerate(grams)}
    ex.f_grams = set(grams)
    toks, lens = vocab_arrays(ex, max_n)
    B, L = 8, 64
    q = zipf_tokens(rng, B * L, V, a=1.15).reshape(B, L).astype(np.int64)
    # plant vocabulary f-grams so most positions hit
    for b in range(B):
        i = 0
        while i < L:
            if rng.random() < 0.7:
                g = grams[int(rng.integers(0, N))]
                n = min(len(g), L - i)
                q[b, i:i + n] = g[:n]
                i += n
            else:
                i += 1
    fid, ml = ref_longest_batch(ex, q)
    np.savez_compressed(os.path.join(HERE, "vocab_n5.npz"), vocab_tokens=toks, vocab_lens=lens, max_n=max_n,
                        query=q, fgram_id=fid, match_len=ml)


def make_cache_small():
    rng = np.random.default_rng(99)
    torch.manual_seed(99)
    V, max_n = 40, 3
    corpus = [zipf_tokens(rng, 50, V).tolist() for _ in range(20)]
    ex = NGramExtractor(max_n=max_n, min_freq=2, max_f_grams=200).fit(corpus, verbose=False)
    N, D = len(ex.f_grams), 64
    rows = (torch.randn(N, D) * 0.02).float()
    rows[3] = 0.0                       # an all-zero row (INT8/INT4 scale edge)
    rows[5, 7] = 3.0                    # an outlier
    toks, lens = vocab_arrays(ex, max_n)

    cache = EmbeddingCache(ex, D)
    cache.cache_embeddings(list(range(N)), rows, verbose=False)
    pick = [0, N - 1, 3, 5, 5, 17 % N, 2]
    got = cache.get_embeddings(pick).numpy()

    with tempfile.TemporaryDirectory() as td:
        mm = EmbeddingCache(ex, D, cache_dir=td, use_memory_map=True)
        mm.cache_embeddings(list(range(N)), rows, verbose=False)
        got_mm = mm.get_embeddings(pick).numpy()
        del mm
    assert np.array_equal(got, got_mm)

    half_bits = torch.from_numpy(got).half().view(torch.int16).numpy().view(np.uint16)

    # engine.py:235-259 re-enacted on reference objects (the engine module itself needs HF hub)
    q = zipf_tokens(rng, 40, V).tolist()
    tf = ex.get_token_f_grams(q)
    assembled = torch.zeros((1, len(q), D))
    for pos, grams in tf.items():
        if not grams:
            continue
        ids = [ex.f_gram_to_id[g] for g in grams]
        assembled[0, pos] = cache.get_embeddings(ids, None).mean(dim=0)
    # get_token_embeddings (embedding_cache.py:149-181): pos -> [k, D]
    tok_emb = cache.get_token_embeddings(q)
    te_pos = np.array(sorted(tok_emb.keys()), dtype=np.int32)
    te_cnt = np.array([tok_emb[int(p)].shape[0] for p in te_pos], dtype=np.int32)
    te_rows = np.concatenate([tok_emb[int(p)].numpy() for p in te_pos]) if len(te_pos) else np.zeros((0, D), np.float32)
    fid, ml = ref_longest(ex, q)

    # artefacts exactly as the reference writes them (n_gram_extractor.py:128-141, embedding_cache.py:183-203)
    ex.save(os.path.join(HERE, "ref_extractor.npy"))
    small = EmbeddingCache(ex, D)
    keep = list(range(0, N, 3))
    small.cache_embeddings(keep, rows[keep], verbose=False)
    small.save(os.path.join(HERE, "ref_cache.npy"))

    np.savez_compressed(os.path.join(HERE, "cache_small.npz"), vocab_tokens=toks, vocab_lens=lens, max_n=max_n,
                        rows=rows.numpy(), pick=np.array(pick, dtype=np.int64), gathered=got, half_bits=half_bits,
                        query=np.array(q, dtype=np.int64), assembled=assembled.numpy()[0],
                        te_pos=te_pos, te_cnt=te_cnt, te_rows=te_rows, fgram_id=fid, match_len=ml)


def make_live_2024():
    """The inputs of test_live_reference_agrees_with_oracle, drawn the same way there."""
    rng = np.random.default_rng(2024)
    corpus = [((rng.zipf(1.2, size=80) - 1) % 60).tolist() for _ in range(30)]
    q = ((rng.zipf(1.2, size=120) - 1) % 60).tolist()
    max_n, min_freq, max_f = 4, 2, 500
    ex = NGramExtractor(max_n=max_n, min_freq=min_freq, max_f_grams=max_f).fit(corpus, verbose=False)
    toks, lens = vocab_arrays(ex, max_n)
    offs, flat = ref_containing(ex, q)
    np.savez_compressed(os.path.join(HERE, "live_2024.npz"), corpus=np.array(corpus, dtype=np.int64), query=np.array(q, dtype=np.int64),
                        max_n=max_n, min_freq=min_freq, max_f_grams=max_f, vocab_tokens=toks, vocab_lens=lens,
                        cont_offs=offs, cont_flat=flat)


FIXTURES = {"kat0": make_kat0, "fit_small": make_fit_small, "fit_medium": make_fit_medium, "vocab_n5": make_vocab_n5,
            "cache_small": make_cache_small, "live_2024": make_live_2024}


if __name__ == "__main__":
    for name in sys.argv[1:] or list(FIXTURES):
        FIXTURES[name]()
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
