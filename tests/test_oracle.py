"""CPU tests: pin the oracle (py + C) against fixtures generated from the unmodified reference."""

import os

import numpy as np
import pytest

from conftest import GOLDEN, load_golden, vocab_dict
from oracle import py_oracle as po
from oracle import ref_shim
from oracle.c_oracle import COracleIndex, lib as c_lib


def _corpus(z):
    offs = z["corpus_offs"]
    return [z["corpus_flat"][offs[i]:offs[i + 1]].tolist() for i in range(len(offs) - 1)]


# ---- vocabulary construction --------------------------------------------------------------

def test_kat0_fit_and_match():
    z = load_golden("kat0.npz")
    grams = po.fit([[1, 2, 3, 4, 1, 2, 3], [2, 3, 4, 5], [1, 2, 9]], 3, 1, 100)
    expect = [tuple(int(t) for t in z["vocab_tokens"][i, :z["vocab_lens"][i]]) for i in range(len(z["vocab_lens"]))]
    assert grams == expect
    # SURVEY.md 8c KAT-0, literally
    assert grams[:4] == [(2,), (1,), (3,), (1, 2)] and grams[17] == (1, 2, 9)
    _, g2i, _ = po.vocab_maps(grams)
    for fn in (po.longest_match_window, po.longest_match_direct):
        fid, ml = fn(g2i, 3, z["query"].tolist())
        assert fid.tolist() == [1, 3, 7, -1, 1, 3, 7, 8, 14, 15, 0, 4]
        assert ml.tolist() == [1, 2, 3, 0, 1, 2, 3, 3, 3, 1, 1, 2]
        assert np.array_equal(fid, z["fgram_id"]) and np.array_equal(ml, z["match_len"])
    # truncate-THEN-filter, first-seen tie order (n_gram_extractor.py:91-94)
    assert po.fit([[7, 8, 7, 8, 9]], 2, 2, 3) == [(7,), (8,), (7, 8)]


@pytest.mark.parametrize("name", ["fit_small.npz", "fit_medium.npz"])
def test_fit_small_matches_reference(name):
    """fit_medium: the max_f_grams cut falls inside a run of 594 n-grams with count 3 (first-seen order keeps 583 of them)."""
    z = load_golden(name)
    grams = po.fit(_corpus(z), int(z["max_n"]), int(z["min_freq"]), int(z["max_f_grams"]))
    expect = [tuple(int(t) for t in z["vocab_tokens"][i, :z["vocab_lens"][i]]) for i in range(len(z["vocab_lens"]))]
    assert grams == expect


# ---- match ---------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["fit_small.npz", "vocab_n5.npz"])
def test_longest_match_golden(name):
    z = load_golden(name)
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    max_n = int(z["max_n"])
    for via_window in (True, False):
        fid, ml = po.match_batch(g2i, max_n, z["query"], via_window=via_window)
        assert np.array_equal(fid, z["fgram_id"])
        assert np.array_equal(ml, z["match_len"])
    cix = COracleIndex(z["vocab_tokens"], z["vocab_lens"])
    for nt in (1, 3):
        fid, ml = cix.match(z["query"], nthreads=nt)
        assert np.array_equal(fid, z["fgram_id"]) and np.array_equal(ml, z["match_len"])
    all_py = po.match_all_batch(g2i, max_n, z["query"])
    assert np.array_equal(cix.match_all(z["query"], nthreads=2), all_py)
    # longest = highest n present in match_all
    has = all_py >= 0
    ml2 = np.where(has.any(-1), max_n - np.argmax(has[..., ::-1], axis=-1), 0)
    assert np.array_equal(ml2.astype(np.uint8), z["match_len"])


def test_containing_lists_golden():
    """get_token_f_grams (all f-grams containing a position, order n asc then start asc)."""
    z = load_golden("fit_small.npz")
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    for b in range(z["query"].shape[0]):
        tf = po.token_f_grams(g2i.keys(), int(z["max_n"]), z["query"][b].tolist())
        flat = z["cont_flat"][z["cont_flat_offs"][b]:z["cont_flat_offs"][b + 1]]
        offs = z["cont_offs"][b]
        for pos in range(z["query"].shape[1]):
            assert [g2i[g] for g in tf[pos]] == flat[offs[pos]:offs[pos + 1]].tolist()


def test_c_oracle_rejects_duplicates_and_handles_edges():
    toks = np.array([[1, 2], [1, 2]], dtype=np.int32)
    with pytest.raises(ValueError):
        COracleIndex(toks, np.array([2, 2], dtype=np.uint8))
    # same tokens, different length = different f-grams
    cix = COracleIndex(np.array([[1, -1], [1, 1]], dtype=np.int32), np.array([1, 2], dtype=np.uint8))
    fid, ml = cix.match(np.array([[1, 1, 1, 5]], dtype=np.int64))
    assert fid.tolist() == [[0, 1, 1, -1]] and ml.tolist() == [[1, 2, 2, 0]]
    # ids outside int32 never match; L = 1; empty batch
    fid, ml = cix.match(np.array([[2 ** 40 + 1]], dtype=np.int64))
    assert fid.tolist() == [[-1]]
    fid, ml = cix.match(np.zeros((0, 7), dtype=np.int64))
    assert fid.shape == (0, 7)
    # empty vocabulary
    e = COracleIndex(np.zeros((0, 3), dtype=np.int32), np.zeros(0, dtype=np.uint8))
    assert e.match(np.array([[1, 2, 3]], dtype=np.int64))[0].tolist() == [[-1, -1, -1]]


def test_fuzz_py_vs_c_oracle():
    rng = np.random.default_rng(5)
    for trial in range(20):
        max_n = int(rng.integers(1, 7))
        V = int(rng.integers(2, 30))
        N = int(rng.integers(1, 200))
        seen, grams = set(), []
        for _ in range(N):
            g = tuple(int(t) for t in rng.integers(0, V, size=int(rng.integers(1, max_n + 1))))
            if g not in seen:
                seen.add(g)
                grams.append(g)
        toks = np.full((len(grams), max_n), -1, np.int32)
        lens = np.zeros(len(grams), np.uint8)
        for i, g in enumerate(grams):
            toks[i, :len(g)] = g
            lens[i] = len(g)
        g2i = {g: i for i, g in enumerate(grams)}
        B, L = int(rng.integers(1, 5)), int(rng.integers(1, 40))
        q = rng.integers(0, V, size=(B, L)).astype(np.int64)
        a = po.match_batch(g2i, max_n, q, via_window=True)
        b = po.match_batch(g2i, max_n, q, via_window=False)
        c = COracleIndex(toks, lens).match(q, nthreads=2)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
        assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1])


def _live_corpus_and_query():
    rng = np.random.default_rng(2024)
    corpus = [((rng.zipf(1.2, size=80) - 1) % 60).tolist() for _ in range(30)]
    return corpus, ((rng.zipf(1.2, size=120) - 1) % 60).tolist()


@pytest.mark.skipif(not (os.path.exists(os.path.join(GOLDEN, "live_2024.npz")) or ref_shim.available()),
                    reason="needs tests/golden/live_2024.npz or a reference checkout (see tests/golden/make_golden.py)")
def test_live_reference_agrees_with_oracle():
    """fit and get_token_f_grams of the unmodified reference on one more seeded corpus and query: against its output stored
    by tests/golden/make_golden.py, and side by side with the reference itself when a checkout is present."""
    corpus, q = _live_corpus_and_query()
    grams = po.fit(corpus, 4, 2, 500)
    tf = po.token_f_grams(set(grams), 4, q)
    if os.path.exists(os.path.join(GOLDEN, "live_2024.npz")):
        z = load_golden("live_2024.npz")
        assert np.array_equal(z["corpus"], corpus) and np.array_equal(z["query"], q)
        assert grams == [tuple(int(t) for t in z["vocab_tokens"][i, :z["vocab_lens"][i]]) for i in range(len(z["vocab_lens"]))]
        g2i = {g: i for i, g in enumerate(grams)}
        offs = z["cont_offs"]
        for pos in range(len(q)):
            assert [g2i[g] for g in tf[pos]] == z["cont_flat"][offs[pos]:offs[pos + 1]].tolist()
    if ref_shim.available():
        NGramExtractor, EmbeddingCache = ref_shim.load_reference()
        ex = NGramExtractor(max_n=4, min_freq=2, max_f_grams=500).fit(corpus, verbose=False)
        assert grams == [ex.id_to_f_gram[i] for i in range(len(grams))] and len(grams) == len(ex.f_grams)
        assert tf == ex.get_token_f_grams(q)


# ---- rows: gather, fp16 cast, quant formulas ---------------------------------------------------

def test_gather_and_half_cast_golden():
    z = load_golden("cache_small.npz")
    tab = po.OracleTable.from_fp32(z["rows"], "fp16")
    assert np.array_equal(z["gathered"], z["rows"][z["pick"]])          # embedding_cache.py:127-141 is a pure gather
    bits = po.cast_bits(tab.rows_fp32(z["pick"]), "fp16")
    assert np.array_equal(bits, z["half_bits"])                          # engine.py:265-266 `.half()`
    assert np.array_equal(po.f32_to_f16_bits(z["gathered"]), z["half_bits"])
    # the unquantised format is the reference's own storage: gathered rows are the fixture bit for bit
    t32 = po.OracleTable.from_fp32(z["rows"], "fp32")
    assert np.array_equal(t32.rows_fp32(z["pick"]).view(np.uint32), z["gathered"].view(np.uint32))


def test_assemble_mean_golden():
    z = load_golden("cache_small.npz")
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    got = po.assemble_mean(g2i, int(z["max_n"]), lambda ids: z["rows"][ids], z["query"].tolist(), z["rows"].shape[1])
    np.testing.assert_allclose(got, z["assembled"], rtol=0, atol=1e-7)
    assert np.array_equal(got.view(np.uint32), z["assembled"].view(np.uint32))     # the engine's tensor, bit for bit
    # ... and so is the kernel's arithmetic (csrc/table.cu mean_kernel): fp32 running sum in list order, one divide
    tf = po.token_f_grams(g2i.keys(), int(z["max_n"]), z["query"].tolist())
    seq = np.zeros_like(got)
    for pos, grams in tf.items():
        acc = np.zeros(got.shape[1], np.float32)
        for g in grams:
            acc = (acc + z["rows"][g2i[g]]).astype(np.float32)
        seq[pos] = (acc / np.float32(len(grams))).astype(np.float32) if len(grams) > 1 else acc
    assert np.array_equal(seq.view(np.uint32), z["assembled"].view(np.uint32))


def test_bf16_f16_casts_against_torch_and_c():
    import torch
    rng = np.random.default_rng(0)
    x = np.concatenate([
        rng.standard_normal(4000).astype(np.float32) * 0.02,
        rng.standard_normal(2000).astype(np.float32) * 1e-6,
        rng.standard_normal(2000).astype(np.float32) * 7e4,
        np.array([0.0, -0.0, np.inf, -np.inf, 65504.0, 65519.99, 65520.0, 2 ** -24, 2 ** -25, 2 ** -25 * 1.0001,
                  1.0009765625, 1.00048828125, 1.00146484375, 3.0e-5, 6.1e-5, 5.96e-8], dtype=np.float32),
        np.arange(0, 70000, 7, dtype=np.uint32).astype(np.float32) / 1024.0,
    ])
    t = torch.from_numpy(x)
    bf = t.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)
    hf = t.to(torch.float16).view(torch.int16).numpy().view(np.uint16)
    assert np.array_equal(po.f32_to_bf16_bits(x), bf)
    assert np.array_equal(po.f32_to_f16_bits(x), hf)
    L = c_lib()
    assert np.array_equal(np.array([L.oracle_f32_to_bf16(float(v)) for v in x], dtype=np.uint16), bf)
    assert np.array_equal(np.array([L.oracle_f32_to_f16(float(v)) for v in x], dtype=np.uint16), hf)
    allh = np.arange(0, 65536, dtype=np.uint16)
    finite = (allh & 0x7C00) != 0x7C00
    back = np.array([L.oracle_f16_to_f32(int(h)) for h in allh[finite]], dtype=np.float32)
    assert np.array_equal(back, allh[finite].view(np.float16).astype(np.float32))
    assert np.array_equal(po.bf16_bits_to_f32(bf), t.to(torch.bfloat16).float().numpy())


def test_quant_formulas_properties():
    rng = np.random.default_rng(3)
    rows = (rng.standard_normal((64, 256)) * 0.02).astype(np.float32)
    rows[3] = 0
    rows[5, 7] = 3.0
    q, s = po.quant_int8_row(rows)
    assert s[3] == 1.0 and not q[3].any()
    assert np.abs(q).max() <= 127 and np.all(np.abs(q).max(axis=1)[np.arange(64) != 3] == 127)
    dq = po.dequant_int8_row(q, s)
    assert np.all(np.abs(dq - rows) <= s[:, None] * 0.5 * (1 + 1e-6))
    p, s16 = po.quant_int4_group(rows, 128)
    assert p.shape == (64, 128) and s16.shape == (64, 2) and s16.dtype == np.float16
    assert np.all(s16[3] == 1.0)
    assert ((p & 0xF) >= 1).all() and ((p >> 4) >= 1).all()              # nibble 0 (= -8) never produced
    dq4 = po.dequant_int4_group(p, s16, 128)
    sw = np.repeat(s16.astype(np.float32), 128, axis=1)
    # |error| <= half a step, except where the fp16-rounded scale is below max/7 and the clamp bites
    assert np.all(np.abs(dq4 - rows) <= sw * 0.5 * 1.01 + np.abs(rows) * 2e-3)
    assert np.array_equal(po.unpack_int4(p)[:, 0::2], (p & 0xF).astype(np.int8) - 8)


@pytest.mark.parametrize("quant", ["fp32", "fp16", "int8", "int4"])
@pytest.mark.parametrize("out_dtype", ["bf16", "fp16"])
def test_embed_forward_py_vs_c(quant, out_dtype):
    from scone_b200.utils.synthetic import pack_table_numpy
    z = load_golden("vocab_n5.npz")
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    rng = np.random.default_rng(11)
    N, D, V = len(g2i), 256, 300
    rows = (rng.standard_normal((N, D)) * 0.02).astype(np.float32)
    base = po.cast_bits((rng.standard_normal((V, D)) * 0.02).astype(np.float32), out_dtype)
    tab = po.OracleTable.from_fp32(rows, quant)
    out, fid, ml = po.embed_forward(g2i, int(z["max_n"]), tab, base, z["query"], out_dtype)
    assert np.array_equal(fid, z["fgram_id"]) and np.array_equal(ml, z["match_len"])
    packed, row_stride, scale_off = pack_table_numpy(tab.quant, tab.payload, tab.scales)
    cix = COracleIndex(z["vocab_tokens"], z["vocab_lens"])
    scales = packed[:, scale_off:] if scale_off else None
    cout, cid, clen, err = cix.embed(quant, D, 128, packed, row_stride, scales, row_stride, base, z["query"], out_dtype,
                                     nthreads=2)
    assert err == 0
    assert np.array_equal(cid, fid) and np.array_equal(clen, ml)
    assert np.array_equal(cout, out)


@pytest.mark.parametrize("out_dtype", ["bf16", "fp16"])
def test_embed_forward_additive_is_the_reference_combine(out_dtype):
    """additive=True restates `combined = base_embeddings + f_gram_embeddings` then `+ position_embeddings`
    (language_model.py:239-254): checked against the same expression evaluated by torch in fp32 on the 16-bit inputs."""
    import torch
    z = load_golden("vocab_n5.npz")
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    rng = np.random.default_rng(5)
    N, D, V = len(g2i), 64, 300
    q = z["query"]
    rows = (rng.standard_normal((N, D)) * 0.02).astype(np.float32)
    base = po.cast_bits((rng.standard_normal((V, D)) * 0.02).astype(np.float32), out_dtype)
    pos = po.cast_bits((rng.standard_normal((q.shape[1], D)) * 0.01).astype(np.float32), out_dtype)
    tab = po.OracleTable.from_fp32(rows, "fp16")
    tdt = torch.bfloat16 if out_dtype == "bf16" else torch.float16
    as_t = lambda bits: torch.from_numpy(bits.view(np.int16).copy()).view(tdt).float()
    for with_pos in (False, True):
        out, fid, ml = po.embed_forward(g2i, int(z["max_n"]), tab, base, q, out_dtype, pos_emb_bits=pos if with_pos else None,
                                        additive=True)
        assert np.array_equal(fid, z["fgram_id"])
        fg = torch.zeros(q.shape + (D,))                                    # engine.py:238: zeros where no f-gram
        hit = torch.from_numpy(fid >= 0)
        fg[hit] = torch.from_numpy(tab.rows_fp32(fid[fid >= 0]))
        combined = as_t(base)[torch.from_numpy(q)] + fg                     # language_model.py:239-243
        if with_pos:
            combined = combined + as_t(pos)[None]                           # language_model.py:253-254
        want = combined.to(tdt).view(torch.int16).numpy().view(np.uint16)
        assert np.array_equal(out, want)
        plain, _, _ = po.embed_forward(g2i, int(z["max_n"]), tab, base, q, out_dtype, pos_emb_bits=pos if with_pos else None)
        assert np.array_equal(plain[fid < 0], out[fid < 0])                 # misses: identical to replace mode


@pytest.mark.parametrize("quant", ["fp16", "int8", "int4"])
@pytest.mark.parametrize("out_dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("with_pos,additive", [(True, False), (False, True), (True, True)])
def test_embed_forward_modes_py_vs_c(quant, out_dtype, with_pos, additive):
    """The position add and the additive combine: the C restatement (used at sizes the Python one cannot reach) agrees
    with the Python one bit for bit, including a token outside the base table (zero base row + error flag)."""
    from scone_b200.utils.synthetic import pack_table_numpy
    z = load_golden("vocab_n5.npz")
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    rng = np.random.default_rng(17)
    N, D, V = len(g2i), 128, 300
    q = z["query"]
    rows = (rng.standard_normal((N, D)) * 0.02).astype(np.float32)
    base = po.cast_bits((rng.standard_normal((V, D)) * 0.02).astype(np.float32), out_dtype)
    pos = po.cast_bits((rng.standard_normal((q.shape[1] + 3, D)) * 0.01).astype(np.float32), out_dtype) if with_pos else None
    tab = po.OracleTable.from_fp32(rows, quant)
    out, fid, ml = po.embed_forward(g2i, int(z["max_n"]), tab, base, q, out_dtype, pos_emb_bits=pos, additive=additive)
    packed, row_stride, scale_off = pack_table_numpy(tab.quant, tab.payload, tab.scales)
    cix = COracleIndex(z["vocab_tokens"], z["vocab_lens"])
    scales = packed[:, scale_off:] if scale_off else None
    cout, cid, clen, err = cix.embed(quant, D, 128, packed, row_stride, scales, row_stride, base, q, out_dtype, nthreads=3,
                                     pos_bits=pos, additive=additive)
    assert err == 0 and np.array_equal(cid, fid) and np.array_equal(clen, ml)
    assert np.array_equal(cout, out)
    assert (fid >= 0).any() and (fid < 0).any()


# ---- property-based fuzz (SURVEY.md section 4: hypothesis over vocabularies / sequences / max_n) --------------------------

from hypothesis import given, settings, strategies as st  # noqa: E402


@settings(max_examples=60, deadline=None)
@given(st.data())
def test_hypothesis_match_py_window_vs_direct_vs_c(data):
    max_n = data.draw(st.integers(1, 7))
    V = data.draw(st.integers(1, 12))
    grams = data.draw(st.lists(st.lists(st.integers(0, V - 1), min_size=1, max_size=max_n).map(tuple), max_size=40, unique=True))
    rows = data.draw(st.lists(st.lists(st.integers(0, V), min_size=1, max_size=30), min_size=1, max_size=4))
    L = max(len(r) for r in rows)
    q = np.array([r + [V] * (L - len(r)) for r in rows], dtype=np.int64)      # V = a token outside the vocabulary as pad
    g2i = {g: i for i, g in enumerate(grams)}
    toks = np.full((len(grams), max_n), -1, np.int32)
    lens = np.zeros(len(grams), np.uint8)
    for i, g in enumerate(grams):
        toks[i, :len(g)] = g
        lens[i] = len(g)
    a = po.match_batch(g2i, max_n, q, via_window=True)
    b = po.match_batch(g2i, max_n, q, via_window=False)
    c = COracleIndex(toks, lens).match(q, nthreads=2)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[0], c[0]) and np.array_equal(a[1], c[1])
    # a match is a real f-gram ending there, and nothing longer in the vocabulary ends there
    for bi in range(q.shape[0]):
        for i in range(L):
            n = int(a[1][bi, i])
            if n:
                assert g2i[tuple(q[bi, i - n + 1:i + 1].tolist())] == a[0][bi, i]
            for m in range(n + 1, min(max_n, i + 1) + 1):
                assert tuple(q[bi, i - m + 1:i + 1].tolist()) not in g2i


@settings(max_examples=40, deadline=None)
@given(st.integers(0, 2 ** 32 - 1), st.sampled_from(["fp16", "int8", "int4"]), st.sampled_from(["bf16", "fp16"]))
def test_hypothesis_dequant_py_vs_c(seed, quant, out_dtype):
    from scone_b200.utils.synthetic import pack_table_numpy
    rng = np.random.default_rng(seed)
    D = 128 * int(rng.integers(1, 4))
    rows = (rng.standard_normal((5, D)) * float(10.0 ** rng.uniform(-6, 3))).astype(np.float32)
    rows[int(rng.integers(0, 5))] = 0
    tab = po.OracleTable.from_fp32(rows, quant)
    packed, stride, soff = pack_table_numpy(quant, tab.payload, tab.scales)
    toks = np.arange(5, dtype=np.int32).reshape(5, 1)
    cix = COracleIndex(toks, np.ones(5, np.uint8))
    base = np.zeros((6, D), np.uint16)
    q = np.arange(6, dtype=np.int64).reshape(1, 6)
    out, fid, _, err = cix.embed(quant, D, 128, packed, stride, packed[:, soff:] if soff else None, stride, base, q, out_dtype)
    assert err == 0 and fid.tolist() == [[0, 1, 2, 3, 4, -1]]
    assert np.array_equal(out[0, :5], po.cast_bits(tab.rows_fp32(np.arange(5)), out_dtype))


def test_fold_projection_contract():
    """oracle/py_oracle.py::fold_projection -- the reference's bias-free f_gram_projection (language_model.py:172-176, :236)
    on bf16-rounded inputs: the stated bound must hold for fp32 accumulation in ANY order (forward, reverse, pairwise, blocked),
    because the tensor cores' order is unspecified; and torch's own Linear on the rounded inputs lands inside it too."""
    import torch
    rng = np.random.default_rng(3)
    rows = (rng.standard_normal((37, 384)) * 0.5).astype(np.float32)
    W = (rng.standard_normal((96, 384)) / np.sqrt(384)).astype(np.float32)
    P, bound = po.fold_projection(rows, W)
    a, w = po.round_to_bf16(rows), po.round_to_bf16(W)
    assert np.array_equal(po.round_to_bf16(a), a) and np.abs(a - rows).max() <= np.abs(rows).max() * 2.0 ** -8
    prods = a[:, None, :] * w[None, :, :]                       # exact in fp32: 8-bit x 8-bit significands
    fwd = np.zeros((37, 96), np.float32)
    for k in range(384):
        fwd = (fwd + prods[:, :, k]).astype(np.float32)
    rev = np.zeros((37, 96), np.float32)
    for k in range(383, -1, -1):
        rev = (rev + prods[:, :, k]).astype(np.float32)
    blocked = prods.reshape(37, 96, 24, 16).sum(axis=3, dtype=np.float32).sum(axis=2, dtype=np.float32)
    for x in (fwd, rev, blocked, prods.sum(axis=2, dtype=np.float32)):
        assert np.all(np.abs(x - P) <= bound)
    lin = torch.nn.functional.linear(torch.from_numpy(a), torch.from_numpy(w)).numpy()         # the reference's op (fp32 Linear)
    assert np.all(np.abs(lin - P) <= bound)
    assert bound.max() < 1e-4 * np.abs(P).max()                 # ... and it is tight enough to mean something
