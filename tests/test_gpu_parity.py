"""GPU parity tests: the CUDA path (through the C ABI) against the oracle, bit-exact.

Bars (BASELINE.json north_star): f-gram ids and match lengths bit-exact; embeddings within 1 ulp
(bf16 / fp16) of the pinned dequant formula -- here they are in fact required to be bit-identical,
with the 1-ulp bound asserted first so a failure says which bar broke.
"""

import numpy as np
import pytest
import torch

from conftest import load_golden, vocab_dict
from oracle import py_oracle as po
from oracle.c_oracle import COracleIndex

pytestmark = pytest.mark.gpu

DEV = "cuda"


@pytest.fixture(autouse=True, params=["auto", "wide", "c20"])
def index_format(request, monkeypatch):
    """Every test runs twice: with the library defaults (compact 16-byte slots whenever the tokens allow; the Bloom
    pre-filter consulted by large batches only; kernel chosen per mode), with the 32-byte slot format forced, the pre-filter
    consulted for every batch size and the single-ring kernel (embed_bulk_kernel) for the plain path, and with the second
    compact slot format preferred and the three-role pipeline kernel (embed_pipe.cuh) for the plain path.  Modes with extra
    rows per position (position add, additive combine) take the pipeline in all three."""
    if request.param == "wide":
        monkeypatch.setenv("SCONE_INDEX_FORMAT", "wide")
        monkeypatch.setenv("SCONE_INDEX_FILTER", "always")
        monkeypatch.setenv("SCONE_EMBED_PIPE", "0")
    elif request.param == "c20":
        # the second compact slot format (five 20-bit tokens; what V = 128 000 vocabularies get) wherever it fits (max_n <= 5)
        monkeypatch.setenv("SCONE_INDEX_FORMAT", "prefer-compact20")
        monkeypatch.setenv("SCONE_INDEX_FILTER", "always")
        monkeypatch.setenv("SCONE_EMBED_PIPE", "1")             # the pipeline kernel for every mode, the plain path included
    else:
        monkeypatch.delenv("SCONE_INDEX_FORMAT", raising=False)
        monkeypatch.delenv("SCONE_INDEX_FILTER", raising=False)
        monkeypatch.delenv("SCONE_EMBED_PIPE", raising=False)
    return request.param


def _mods():
    import scone_b200
    from scone_b200.utils import synthetic
    return scone_b200, synthetic


def _index(toks, lens, **kw):
    sb, _ = _mods()
    return sb.FGramIndex(torch.from_numpy(np.ascontiguousarray(toks, dtype=np.int32)).to(DEV),
                         torch.from_numpy(np.ascontiguousarray(lens, dtype=np.uint8)).to(DEV), **kw)


def _bits(t: torch.Tensor) -> np.ndarray:
    return t.contiguous().view(torch.int16).cpu().numpy().view(np.uint16)


def _from_bits(b: np.ndarray, dtype) -> torch.Tensor:
    return torch.from_numpy(b.view(np.int16).copy()).view(dtype).to(DEV)


TORCH_DT = {"bf16": torch.bfloat16, "fp16": torch.float16}


def test_library_is_native_and_loaded():
    from scone_b200 import _lib
    L = _lib.load()
    assert L.scone_version() == _lib.ABI_VERSION
    before = _lib.launch_count()
    ix = _index(np.array([[1, 2]], np.int32), np.array([2], np.uint8))
    ix.lookup(torch.tensor([[1, 2, 3]], device=DEV))
    torch.cuda.synchronize()
    assert _lib.launch_count() >= before + 3          # build + audit + lookup kernels really launched


# ---- match -------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", ["kat0.npz", "fit_small.npz", "vocab_n5.npz", "cache_small.npz"])
def test_lookup_golden(name):
    z = load_golden(name)
    ix = _index(z["vocab_tokens"], z["vocab_lens"])
    q = z["query"]
    q2 = q[None, :] if q.ndim == 1 else q
    fid, ml = ix.lookup(torch.from_numpy(q2).to(DEV))
    assert np.array_equal(fid.cpu().numpy().reshape(q.shape), z["fgram_id"])
    assert np.array_equal(ml.cpu().numpy().reshape(q.shape), z["match_len"])
    g2i = vocab_dict(z["vocab_tokens"], z["vocab_lens"])
    allm = ix.match_all(torch.from_numpy(q2).to(DEV)).cpu().numpy()
    assert np.array_equal(allm, po.match_all_batch(g2i, z["vocab_tokens"].shape[1], q2))


def test_kat0_literal():
    """SURVEY.md 8c KAT-0 spelled out."""
    sb, _ = _mods()
    ex = sb.NGramExtractor(max_n=3, min_freq=1, max_f_grams=100).fit([[1, 2, 3, 4, 1, 2, 3], [2, 3, 4, 5], [1, 2, 9]], verbose=False)
    assert ex.id_to_f_gram[0] == (2,) and ex.id_to_f_gram[7] == (1, 2, 3) and ex.id_to_f_gram[17] == (1, 2, 9)
    fid, ml = ex.lookup(torch.tensor([[1, 2, 3, 7, 1, 2, 3, 4, 5, 9, 2, 3]], device=DEV))
    assert fid[0].tolist() == [1, 3, 7, -1, 1, 3, 7, 8, 14, 15, 0, 4]
    assert ml[0].tolist() == [1, 2, 3, 0, 1, 2, 3, 3, 3, 1, 1, 2]
    ex2 = sb.NGramExtractor(max_n=2, min_freq=2, max_f_grams=3).fit([[7, 8, 7, 8, 9]], verbose=False)
    assert ex2.f_gram_to_id == {(7,): 0, (8,): 1, (7, 8): 2}


def test_index_build_audit():
    with pytest.raises(ValueError, match="duplicated"):
        _index(np.array([[1, 2], [3, 4], [1, 2]], np.int32), np.array([2, 2, 2], np.uint8))
    with pytest.raises(ValueError, match="lengths"):
        _index(np.array([[1, 2]], np.int32), np.array([3], np.uint8))
    with pytest.raises(ValueError, match="negative"):
        _index(np.array([[1, -1]], np.int32), np.array([2], np.uint8))
    with pytest.raises(ValueError, match="max_n"):
        _index(np.zeros((1, 8), np.int32), np.array([8], np.uint8))
    # same tokens, different length = different keys; empty vocabulary; load factors
    ix = _index(np.array([[1, -1], [1, 1]], np.int32), np.array([1, 2], np.uint8))
    fid, ml = ix.lookup(torch.tensor([[1, 1, 1, 5]], device=DEV))
    assert fid.tolist() == [[0, 1, 1, -1]] and ml.tolist() == [[1, 2, 2, 0]]
    e = _index(np.zeros((0, 3), np.int32), np.zeros((0,), np.uint8))
    assert e.lookup(torch.tensor([[1, 2, 3]], device=DEV))[0].tolist() == [[-1, -1, -1]]
    assert e.len_mask == 0
    # slot format: compact (six 16-bit tokens) when every token < 65535 and max_n <= 6; compact (five 20-bit tokens) when every
    # token < 1048575 and max_n <= 5; 32-byte slots otherwise or when forced
    import os
    fmt = os.environ.get("SCONE_INDEX_FORMAT")
    small = _index(np.array([[1, 2]], np.int32), np.array([2], np.uint8))
    big = _index(np.array([[1, 70000]], np.int32), np.array([2], np.uint8))
    huge = _index(np.array([[1, 1048575]], np.int32), np.array([2], np.uint8))
    long6 = _index(np.array([[1, 70000, 3, 4, 5, 6]], np.int32), np.array([6], np.uint8))
    assert small.slot_format == {"wide": "wide32", "prefer-compact20": "compact20"}.get(fmt, "compact16")
    assert big.slot_format == ("wide32" if fmt == "wide" else "compact20") and big.slot_bytes == (32 if fmt == "wide" else 16)
    assert huge.slot_format == "wide32" and long6.slot_format == "wide32" and huge.slot_bytes == 32
    fid, _ = big.lookup(torch.tensor([[1, 70000, 65535, 1, 70000]], device=DEV))
    assert fid.tolist() == [[-1, 0, -1, -1, 0]]
    fid, _ = big.lookup(torch.tensor([[1, 70000 + (1 << 20), 1, 1048575, 1, 70000]], device=DEV))   # 20-bit aliases must not match
    assert fid.tolist() == [[-1, -1, -1, -1, -1, 0]]
    fid, _ = huge.lookup(torch.tensor([[1, 1048575, 1, 1048574]], device=DEV))
    assert fid.tolist() == [[-1, 0, -1, -1]]
    fid, _ = small.lookup(torch.tensor([[1, 2, 65535, 65536 + 1, 2, 1, 2]], device=DEV))     # 65537 must not alias token 1
    assert fid.tolist() == [[-1, 0, -1, -1, -1, -1, 0]]


def test_lookup_edge_shapes_and_ids():
    _, S = _mods()
    toks, lens = S.make_vocab_numpy(500, 5, 60, seed=4, min_n=1)
    cix = COracleIndex(toks, lens)
    for lf in (0.25, 0.5, 0.9):
        ix = _index(toks, lens, load_factor=lf)
        for (B, L) in [(1, 1), (1, 2), (3, 5), (7, 33), (2, 257), (1, 4096), (33, 1)]:
            q = S.make_stream_numpy(toks, lens, B, L, 60, seed=B * 1000 + L)
            fid, ml = ix.lookup(torch.from_numpy(q).to(DEV))
            rid, rl = cix.match(q)
            assert np.array_equal(fid.cpu().numpy(), rid) and np.array_equal(ml.cpu().numpy(), rl), (lf, B, L)
    # token ids outside int32 / negative: never match, never crash
    q = np.array([[5, 2 ** 40 + 5, -7, 5, 5]], dtype=np.int64)
    fid, ml = ix.lookup(torch.from_numpy(q).to(DEV))
    rid, rl = cix.match(q)
    assert np.array_equal(fid.cpu().numpy(), rid) and np.array_equal(ml.cpu().numpy(), rl)
    # empty batch
    fid, ml = ix.lookup(torch.zeros((0, 9), dtype=torch.long, device=DEV))
    assert fid.shape == (0, 9)
    with pytest.raises(ValueError):
        ix.lookup(torch.zeros((2, 2), dtype=torch.long))          # CPU tensor: no CPU path


@pytest.mark.parametrize("mode", ["never", "always", None])
def test_prefilter_never_changes_a_result(mode, monkeypatch):
    """The Bloom pre-filter has no false negatives: with it off, on for every batch, or on by the size rule (this batch is
    above kFilterMinPositions) the ids and lengths are the C oracle's, bit for bit."""
    sb, S = _mods()
    if mode is None:
        monkeypatch.delenv("SCONE_INDEX_FILTER", raising=False)
    else:
        monkeypatch.setenv("SCONE_INDEX_FILTER", mode)
    N, max_n, V, B, L = 50_000, 5, 3000, 40, 512                    # 20 480 positions
    toks, lens = S.make_vocab_numpy(N, max_n, V, seed=71, min_n=1)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=72, p_plant=0.5)
    ix = _index(toks, lens)
    assert (ix.filter_bytes == 0) == (mode == "never")
    assert ix.filter_bytes in (0, 4 * ((N + 1) // 2 + 31) // 32 * 32) and ix.bytes > ix.filter_bytes      # 16 bits per f-gram
    wid, wlen = COracleIndex(toks, lens).match(q)
    fid, ml = ix.lookup(torch.from_numpy(q).to(DEV))
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    allm = ix.match_all(torch.from_numpy(q[:3]).to(DEV)).cpu().numpy()           # small batch: filter only if "always"
    best = np.where(allm >= 0, np.arange(1, max_n + 1)[None, None, :], 0).max(axis=-1)
    assert np.array_equal(best, wlen[:3])
    ix.close()


@pytest.mark.parametrize("max_n", [1, 2, 3, 4, 5, 6, 7])
def test_lookup_all_max_n(max_n):
    _, S = _mods()
    toks, lens = S.make_vocab_numpy({1: 10, 2: 400}.get(max_n, 3000), max_n, 40, seed=max_n, min_n=1)
    ix = _index(toks, lens)
    q = S.make_stream_numpy(toks, lens, 5, 301, 40, seed=9)
    fid, ml = ix.lookup(torch.from_numpy(q).to(DEV))
    rid, rl = COracleIndex(toks, lens).match(q)
    assert np.array_equal(fid.cpu().numpy(), rid) and np.array_equal(ml.cpu().numpy(), rl)
    assert (rl == max_n).any()


# ---- table formats ---------------------------------------------------------------------------------------------

@pytest.mark.parametrize("quant", ["fp32", "fp16", "int8", "int4", "int4/8", "int4/32", "int4/256"])   # int4/<group>: INT4 groups other than 128
@pytest.mark.parametrize("D", [128, 768, 1024])
def test_table_store_is_bit_identical_to_oracle_quantiser(quant, D):
    sb, S = _mods()
    quant, group = quant.split("/")[0], int(quant.split("/")[1]) if "/" in quant else 128
    if D % group:
        pytest.skip("D must be a multiple of the INT4 group")
    rows = S.make_rows_numpy(300, D, seed=D)
    rows[3] = 0.0
    rows[5, 7] = 3.0
    rows[6] *= 1e-7            # int4: scale underflows fp16 -> scale 1
    rows[7] *= 1e4
    tab = po.OracleTable.from_fp32(rows, quant, group)
    packed, stride, soff = S.pack_table_numpy(quant, tab.payload, tab.scales)
    t = sb.CacheTable(300, D, quant, group=group)
    assert (t.row_stride, t.scale_offset) == (stride, soff)
    perm = np.random.default_rng(0).permutation(300)
    t.store(torch.from_numpy(rows[perm]).to(DEV), torch.from_numpy(perm).to(DEV))
    assert np.array_equal(t.storage.cpu().numpy(), packed)
    # dequantising gather == oracle dequant, exactly, in fp32 and in both 16-bit types
    pick = np.array([0, 299, 3, 5, 5, 6, 7, 17], dtype=np.int64)
    got = t.gather(torch.from_numpy(pick).to(DEV)).cpu().numpy()
    assert np.array_equal(got, tab.rows_fp32(pick))
    for name, dt in TORCH_DT.items():
        got16 = _bits(t.gather(torch.from_numpy(pick).to(DEV), dt))
        assert np.array_equal(got16, po.cast_bits(tab.rows_fp32(pick), name))


# ---- the fused path ------------------------------------------------------------------------------------------------

def _embed_case(quant, out_dtype, D, max_n, N, V, B, L, seed, min_n=2, p_plant=0.7, with_pos=False):
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(N, max_n, V, seed=seed, min_n=min_n)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=seed + 1, p_plant=p_plant)
    rows = S.make_rows_numpy(N, D, seed=seed + 2)
    base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=seed + 3), out_dtype)
    tab = po.OracleTable.from_fp32(rows, quant)
    packed, stride, soff = S.pack_table_numpy(quant, tab.payload, tab.scales)
    cix = COracleIndex(toks, lens)
    want, wid, wlen, err = cix.embed(quant, D, 128, packed, stride, packed[:, soff:] if soff else None, stride, base_bits, q,
                                     out_dtype, nthreads=4)
    assert err == 0
    ix = _index(toks, lens)
    t = sb.CacheTable(N, D, quant)
    t.store(torch.from_numpy(rows).to(DEV))
    base = _from_bits(base_bits, TORCH_DT[out_dtype])
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, torch.from_numpy(q).to(DEV), status=status)
    torch.cuda.synchronize()
    assert np.array_equal(fid.cpu().numpy(), wid), "f-gram ids must be bit-exact"
    assert np.array_equal(ml.cpu().numpy(), wlen), "match lengths must be bit-exact"
    got = _bits(out)
    assert po.ulp_distance(got, want).max() <= 1, "embeddings must be within 1 ulp"
    assert np.array_equal(got, want)
    assert int(status.item()) == 0
    return dict(toks=toks, lens=lens, q=q, tab=tab, base_bits=base_bits, want=want, wid=wid, hit=float((wid >= 0).mean()))


@pytest.mark.parametrize("quant", ["fp32", "fp16", "int8", "int4"])
@pytest.mark.parametrize("out_dtype", ["bf16", "fp16"])
@pytest.mark.parametrize("D,max_n", [(128, 3), (768, 3), (1024, 4), (4096, 5), (2048, 7), (8, 1), (136, 2)])
def test_embed_forward_matches_oracle(quant, out_dtype, D, max_n):
    if quant == "int4" and D % 128:
        pytest.skip("INT4 needs D % group == 0")
    r = _embed_case(quant, out_dtype, D, max_n, N=100 if max_n == 1 else 2000, V=500, B=3, L=211, seed=D + max_n,
                    min_n=1 if max_n < 3 else 2)
    assert 0.2 < r["hit"] < 1.0            # both branches exercised


def test_embed_forward_python_oracle_config1_shape():
    """BASELINE config 1 in full against the PYTHON oracle (the reference-pinned one): D = 768, max_n = 3,
    FP16 table, batch 8 x 512; vocabulary 100 000 f-grams."""
    sb, S = _mods()
    N, D, V, max_n, B, L = 100_000, 768, 50_257, 3, 8, 512
    toks, lens = S.make_vocab_numpy(N, max_n, V, seed=0, min_n=1)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=1)
    rows = S.make_rows_numpy(N, D, seed=2)
    base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=3), "bf16")
    g2i = vocab_dict(toks, lens)
    want, wid, wlen = po.embed_forward(g2i, max_n, po.OracleTable.from_fp32(rows, "fp16"), base_bits, q, "bf16")
    # the window form of the reference primitive on a sample of rows
    w2, l2 = po.match_batch(g2i, max_n, q[:2], via_window=True)
    assert np.array_equal(w2, wid[:2]) and np.array_equal(l2, wlen[:2])
    ex = sb.NGramExtractor.from_arrays(toks, lens)
    cache = sb.EmbeddingCache(ex, D, quant="fp16", out_dtype=torch.bfloat16)
    cache.cache_embeddings(list(range(N)), torch.from_numpy(rows), verbose=False)
    cache.set_base_embedding(_from_bits(base_bits, torch.bfloat16))
    out, fid, ml = cache.lookup(torch.from_numpy(q).to(DEV))
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    assert np.array_equal(_bits(out), want)
    assert cache.status() == 0
    assert (wid >= 0).mean() > 0.5


def test_embed_forward_status_and_fallback_edges():
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(100, 3, 50, seed=1)
    ix = _index(toks, lens)
    t = sb.CacheTable(100, 64, "int8")
    t.store(torch.from_numpy(S.make_rows_numpy(100, 64)).to(DEV))
    base = torch.randn(50, 64, device=DEV).to(torch.bfloat16)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    q = torch.tensor([[49, 50, 7, -1, 3]], device=DEV)       # 50 and -1 are outside the base table
    out, fid, ml = sb.embed_forward(ix, t, base, q, status=status)
    assert int(status.item()) == 1
    miss = (fid[0] < 0).cpu().numpy()
    assert miss[1] and miss[3]
    assert not out[0, 1].any() and not out[0, 3].any()         # zero rows, flagged
    assert torch.equal(out[0, 0], base[49]) or not miss[0]
    # empty batch, wrong device / dtype
    o, f, m = sb.embed_forward(ix, t, base, torch.zeros((0, 4), dtype=torch.long, device=DEV))
    assert o.shape == (0, 4, 64)
    with pytest.raises(ValueError):
        sb.embed_forward(ix, t, base.float(), q)
    with pytest.raises(ValueError):
        sb.embed_forward(ix, t, base, q.cpu())


def test_embed_forward_with_positions():
    """Fused wpe add (language_model.py:253-254): fp32(row) + fp32(pos), one RNE rounding."""
    sb, S = _mods()
    # L = 97: tiles straddle the end of a sequence; L = 3 / 1: a tile spans several sequences (its position rows are several blocks)
    # max_n = 1 / 2: 32 / 16 positions per tile (with 32 the lane that stages the position block also stages a row)
    for quant, out_dtype, B, L, max_n in (("int8", "bf16", 4, 97, 4), ("fp16", "fp16", 4, 97, 4), ("int4", "bf16", 4, 97, 4), ("int8", "bf16", 41, 3, 4),
                                          ("fp32", "bf16", 37, 1, 4), ("fp16", "bf16", 9, 50, 1), ("int8", "fp16", 7, 45, 2), ("fp32", "bf16", 30, 5, 1)):
        N, D, V = (1000, 256, 300) if max_n > 1 else (60, 256, 300)
        toks, lens = S.make_vocab_numpy(N, max_n, V, seed=21, min_n=min(2, max_n))
        q = S.make_stream_numpy(toks, lens, B, L, V, seed=22, p_plant=0.7)
        rows = S.make_rows_numpy(N, D, seed=23)
        base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=24), out_dtype)
        pos_bits = po.cast_bits(S.make_rows_numpy(128, D, seed=5), out_dtype)
        want, wid, wlen = po.embed_forward(vocab_dict(toks, lens), max_n, po.OracleTable.from_fp32(rows, quant), base_bits, q,
                                           out_dtype, pos_emb_bits=pos_bits)
        ix = _index(toks, lens)
        t = sb.CacheTable(N, D, quant)
        t.store(torch.from_numpy(rows).to(DEV))
        dt = TORCH_DT[out_dtype]
        out, fid, ml = sb.embed_forward(ix, t, _from_bits(base_bits, dt), torch.from_numpy(q).to(DEV), pos_emb=_from_bits(pos_bits, dt))
        assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
        assert np.array_equal(_bits(out), want)


@pytest.mark.parametrize("quant,out_dtype,D,max_n,with_pos", [
    ("int8", "bf16", 256, 4, False), ("int8", "bf16", 1024, 4, True), ("fp16", "fp16", 768, 3, False), ("fp16", "fp16", 136, 2, True),
    ("int4", "bf16", 4096, 5, False), ("int4", "fp16", 2048, 5, True), ("fp16", "bf16", 4096, 5, True),
    ("fp16", "bf16", 16384, 3, True),            # too wide for a ring: register-load variant
])
def test_embed_forward_additive_combine(quant, out_dtype, D, max_n, with_pos):
    """combine="add": the reference code's `base_embeddings + f_gram_embeddings` (language_model.py:239-243) fused into
    the kernel: (fp32(wte row) + fp32(f-gram row)) [+ fp32(wpe row)], one RNE rounding; misses are the wte row."""
    sb, S = _mods()
    N, V, B, L = 1500, 300, 3, 131
    toks, lens = S.make_vocab_numpy(N, max_n, V, seed=41 + D, min_n=1 if max_n < 3 else 2)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=42, p_plant=0.6)
    rows = S.make_rows_numpy(N, D, seed=43)
    base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=44), out_dtype)
    pos_bits = po.cast_bits(S.make_rows_numpy(L + 5, D, seed=45), out_dtype) if with_pos else None
    want, wid, wlen = po.embed_forward(vocab_dict(toks, lens), max_n, po.OracleTable.from_fp32(rows, quant), base_bits, q,
                                       out_dtype, pos_emb_bits=pos_bits, additive=True)
    assert 0.2 < (wid >= 0).mean() < 1.0
    ix = _index(toks, lens)
    t = sb.CacheTable(N, D, quant)
    t.store(torch.from_numpy(rows).to(DEV))
    dt = TORCH_DT[out_dtype]
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, _from_bits(base_bits, dt), torch.from_numpy(q).to(DEV),
                                    pos_emb=_from_bits(pos_bits, dt) if with_pos else None, status=status, combine="add")
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    got = _bits(out)
    assert po.ulp_distance(got, want).max() <= 1
    assert np.array_equal(got, want)
    assert int(status.item()) == 0
    # replace mode on the same inputs differs exactly where an f-gram ends
    out_r, _, _ = sb.embed_forward(ix, t, _from_bits(base_bits, dt), torch.from_numpy(q).to(DEV),
                                   pos_emb=_from_bits(pos_bits, dt) if with_pos else None)
    same = (_bits(out_r) == got).all(axis=-1)
    assert same[wid < 0].all()
    with pytest.raises(ValueError):
        sb.embed_forward(ix, t, _from_bits(base_bits, dt), torch.from_numpy(q).to(DEV), combine="mean")


def test_embed_forward_additive_token_outside_base_table():
    """A hit whose own token has no base row: the f-gram row alone is written and the status bit is set."""
    sb, S = _mods()
    toks = np.array([[5, 60]], np.int32)
    lens = np.array([2], np.uint8)
    ix = _index(toks, lens)
    t = sb.CacheTable(1, 64, "fp16")
    rows = S.make_rows_numpy(1, 64, seed=1)
    t.store(torch.from_numpy(rows).to(DEV))
    base = torch.from_numpy(S.make_rows_numpy(50, 64, seed=2)).to(DEV).to(torch.float16)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    q = torch.tensor([[5, 60, 7]], device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, q, status=status, combine="add")
    assert fid[0].tolist() == [-1, 0, -1] and int(status.item()) == 1
    assert torch.equal(out[0, 1], torch.from_numpy(rows[0]).half().to(DEV))
    assert torch.equal(out[0, 0], base[5]) and torch.equal(out[0, 2], base[7])


def test_embed_gather_resolved_ids():
    sb, S = _mods()
    r = _embed_case("int4", "fp16", 512, 5, N=1500, V=400, B=2, L=300, seed=31)
    t = sb.CacheTable(1500, 512, "int4")
    t.store(torch.from_numpy(S.make_rows_numpy(1500, 512, seed=33)).to(DEV))
    base = _from_bits(r["base_bits"], torch.float16)
    out = sb.embed_gather(t, base, torch.from_numpy(r["q"]).to(DEV), torch.from_numpy(r["wid"]).to(DEV))
    assert np.array_equal(_bits(out), r["want"])


# ---- full BASELINE sizes: C oracle on everything + size-independent properties -------------------------------------

def test_config2_full_size_against_c_oracle():
    """BASELINE config 2: D = 1024, 1 M f-grams, max_n = 4, INT8, batch 64 x 1024."""
    sb, S = _mods()
    N, D, V, max_n, B, L = 1_000_000, 1024, 50_257, 4, 64, 1024
    toks_d, lens_d = S.make_vocab_device(N, max_n, V, seed=0, device=DEV)
    ix = sb.FGramIndex(toks_d, lens_d)
    q_d = S.make_stream_device(toks_d, lens_d, B, L, V, seed=1)
    t = sb.CacheTable(N, D, "int8")
    S.fill_table_device(t, seed=2)
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, q_d)
    torch.cuda.synchronize()
    toks, lens, q = toks_d.cpu().numpy(), lens_d.cpu().numpy(), q_d.cpu().numpy()
    cix = COracleIndex(toks, lens)
    packed = t.storage.cpu().numpy()
    want, wid, wlen, err = cix.embed("int8", D, 128, packed, t.row_stride, packed[:, t.scale_offset:], t.row_stride,
                                     _bits(base), q, "bf16", nthreads=8)
    assert err == 0
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    assert np.array_equal(_bits(out), want)
    hit = wid >= 0
    assert 0.6 < hit.mean() < 1.0
    # properties that do not depend on the oracle:
    #  (1) a hit row dequantises to the table row it names; a miss row IS the base row
    assert torch.equal(out[torch.from_numpy(~hit).to(DEV)], base[q_d[torch.from_numpy(~hit).to(DEV)]])
    sel = torch.from_numpy(np.flatnonzero(hit.ravel())[:4096]).to(DEV)
    assert torch.equal(out.view(-1, D)[sel], t.gather(fid.view(-1)[sel].long(), torch.bfloat16))
    #  (2) the matched f-gram really is the suffix of the window, and no longer f-gram of the vocabulary was planted there
    ids_flat, wl = q.reshape(-1), wlen.reshape(-1)
    for tpos in np.flatnonzero(hit.ravel())[:2000]:
        n = int(wl[tpos])
        assert np.array_equal(toks[wid.ravel()[tpos], :n], ids_flat[tpos - n + 1:tpos + 1])
    #  (3) idempotence / determinism: a second launch gives identical bits
    out2, fid2, _ = sb.embed_forward(ix, t, base, q_d)
    assert torch.equal(out, out2) and torch.equal(fid, fid2)
    #  (4) row independence: shuffling batch rows shuffles outputs
    perm = torch.randperm(B, device=DEV)
    out3, _, _ = sb.embed_forward(ix, t, base, q_d[perm].contiguous())
    assert torch.equal(out3, out[perm])


# ---- drop-in classes (the reference's own tests, on integer ids) -------------------------------------------------------

def test_dropin_get_token_f_grams_golden():
    sb, _ = _mods()
    z = load_golden("fit_small.npz")
    ex = sb.NGramExtractor.from_arrays(z["vocab_tokens"], z["vocab_lens"])
    g2i = ex.f_gram_to_id
    for b in range(z["query"].shape[0]):
        tf = ex.get_token_f_grams(z["query"][b].tolist())
        flat = z["cont_flat"][z["cont_flat_offs"][b]:z["cont_flat_offs"][b + 1]]
        offs = z["cont_offs"][b]
        for pos in range(z["query"].shape[1]):
            assert [g2i[g] for g in tf[pos]] == flat[offs[pos]:offs[pos + 1]].tolist()


def test_dropin_embedding_cache_like_reference_tests(tmp_path):
    """tests/test_embedding_cache.py of the reference, on the golden cache fixture."""
    sb, _ = _mods()
    z = load_golden("cache_small.npz")
    ex = sb.NGramExtractor.from_arrays(z["vocab_tokens"], z["vocab_lens"])
    N, D = z["rows"].shape
    cache = sb.EmbeddingCache(n_gram_extractor=ex, embedding_dim=D, cache_dir=str(tmp_path / "cache"))
    assert cache.n_gram_extractor is ex and cache.embedding_dim == D
    assert cache.embeddings == {} and cache.memory_mapped_embeddings is None           # :66-72
    rows = torch.from_numpy(z["rows"])
    cache.cache_embeddings({i: rows[i] for i in range(N)})                               # dict form, :75-86
    assert len(cache.embeddings) == N and 5 in cache.embeddings
    got = cache.get_embeddings(z["pick"].tolist())                                      # :89-101
    assert got.dtype == torch.float32 and got.device.type == "cpu"
    assert np.array_equal(got.numpy().view(np.uint32), z["gathered"].view(np.uint32))   # fp32 rows, bit for bit (:132-135)
    assert np.array_equal(got.half().view(torch.int16).numpy().view(np.uint16), z["half_bits"])   # engine.py:265-266
    te = cache.get_token_embeddings(z["query"].tolist())                                # :104-117, with values
    assert sorted(te) == z["te_pos"].tolist()
    assert [te[int(p)].shape[0] for p in z["te_pos"]] == z["te_cnt"].tolist()
    assert np.array_equal(torch.cat([te[int(p)] for p in z["te_pos"]]).numpy().view(np.uint32), z["te_rows"].view(np.uint32))
    # quantised storage is an option of this implementation, not the default: FP16 rows = the reference's rows `.half()`
    c16 = sb.EmbeddingCache(ex, D, quant="fp16")
    c16.cache_embeddings(list(range(N)), rows, verbose=False)
    assert torch.equal(c16.get_embeddings(z["pick"].tolist()), torch.from_numpy(z["gathered"]).half().float())
    with pytest.raises(KeyError):
        sb.EmbeddingCache(ex, D).get_embeddings([0])
    path = tmp_path / "embeddings.cache"
    cache.save(str(path))                                                               # :120-143
    loaded = sb.EmbeddingCache.load(str(path), n_gram_extractor=ex, cache_dir=cache.cache_dir)
    assert len(loaded.embeddings) == N
    assert torch.equal(loaded.get_embeddings(z["pick"].tolist()), got)
    # memory-mapped flavour = offloaded (pinned host) tier, :146-194
    mm = sb.EmbeddingCache(ex, D, cache_dir=str(tmp_path / "cache"), use_memory_map=True)
    with pytest.raises(ValueError):
        sb.EmbeddingCache(ex, D, use_memory_map=True).cache_embeddings([0], rows[:1])
    mm.cache_embeddings(list(range(N)), rows, verbose=False)
    assert isinstance(mm.memory_mapped_embeddings, np.ndarray) and mm.memory_mapped_embeddings.shape == (N, D)
    assert mm.memory_mapped_embeddings.dtype == np.float32 and np.array_equal(mm.memory_mapped_embeddings, z["rows"])   # :84-91
    assert torch.equal(mm.get_embeddings(z["pick"].tolist()), got)
    mm.set_base_embedding(torch.zeros(64, D))
    cache.set_base_embedding(torch.zeros(64, D))
    q = torch.from_numpy(z["query"])[None].to(DEV)
    a, b = mm.lookup(q), cache.lookup(q)
    assert torch.equal(a[0], b[0]) and np.array_equal(a[1].cpu().numpy()[0], z["fgram_id"])


def test_dropin_extractor_save_load_and_fit(tmp_path):
    sb, _ = _mods()
    z = load_golden("fit_small.npz")
    offs = z["corpus_offs"]
    corpus = [z["corpus_flat"][offs[i]:offs[i + 1]].tolist() for i in range(len(offs) - 1)]
    ex = sb.NGramExtractor(max_n=int(z["max_n"]), min_freq=int(z["min_freq"]), max_f_grams=int(z["max_f_grams"]))
    assert ex.fit(corpus, verbose=False) is ex
    t, l = ex.vocab_arrays()
    assert np.array_equal(t, z["vocab_tokens"]) and np.array_equal(l, z["vocab_lens"])   # same ids as the reference fit
    p = str(tmp_path / "ex.npy")
    ex.save(p)
    ex2 = sb.NGramExtractor.load(p)
    assert ex2.f_gram_to_id == ex.f_gram_to_id and ex2.max_n == ex.max_n
    fid, ml = ex2.lookup(torch.from_numpy(z["query"]).to(DEV))
    assert np.array_equal(fid.cpu().numpy(), z["fgram_id"]) and np.array_equal(ml.cpu().numpy(), z["match_len"])


def test_input_embedding_module():
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(800, 3, 200, seed=3)
    ex = sb.NGramExtractor.from_arrays(toks, lens)
    cache = sb.EmbeddingCache(ex, 128, quant="int8", out_dtype=torch.float16)
    cache.cache_embeddings(list(range(800)), torch.from_numpy(S.make_rows_numpy(800, 128)), verbose=False)
    wte, wpe = torch.randn(200, 128) * 0.02, torch.randn(64, 128) * 0.01
    mod = sb.SconeInputEmbedding(cache, wte, wpe)
    q = torch.from_numpy(S.make_stream_numpy(toks, lens, 4, 64, 200)).to(DEV)
    emb, fid, ml = mod(q, return_match=True)
    plain, fid2, _ = cache.lookup(q)
    assert emb.shape == (4, 64, 128) and emb.dtype == torch.float16 and torch.equal(fid, fid2)
    want = (plain.float() + wpe.to(DEV).half().float()[None]).half()
    assert (emb.float() - want.float()).abs().max() <= 2e-4      # single vs double rounding: <= 1 fp16 ulp at this scale
    # combine="add": the reference code's wte + f-gram row + wpe (language_model.py:239-254), one kernel
    mod_add = sb.SconeInputEmbedding(cache, wte, wpe, combine="add")
    emb_add = mod_add(q)
    rows16 = cache.table.gather(fid.clamp(min=0).reshape(-1).long(), torch.float32).reshape(4, 64, 128)
    wte16 = wte.to(DEV).half().float()[q]
    want_add = (wte16 + torch.where((fid >= 0)[..., None], rows16, torch.zeros_like(rows16)) + wpe.to(DEV).half().float()[None]).half()
    assert torch.equal(emb_add, want_add)


# ---- row-sharded tier on one GPU (world size 1 over NCCL: exercises CudaOps end to end) ------------------------------

def test_sharded_tier_world1_nccl():
    import os
    import torch.distributed as dist
    sb, S = _mods()
    from scone_b200 import sharded
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29611")
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device(DEV, 0))
    try:
        for quant in ("int4", "fp16"):
            N, D, V, max_n, B, L = 4000, 512, 300, 5, 3, 130
            toks, lens = S.make_vocab_numpy(N, max_n, V, seed=41)
            q = S.make_stream_numpy(toks, lens, B, L, V, seed=42)
            rows = S.make_rows_numpy(N, D, seed=43)
            base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=44), "bf16")
            want, wid, wlen = po.embed_forward(vocab_dict(toks, lens), max_n, po.OracleTable.from_fp32(rows, quant), base_bits, q, "bf16")
            ix = _index(toks, lens)
            t = sb.CacheTable(N, D, quant)
            t.store(torch.from_numpy(rows).to(DEV))
            cache = sharded.ShardedEmbeddingCache(sharded.CudaOps(ix, t, _from_bits(base_bits, torch.bfloat16)))
            emb, fid, ml = cache.lookup(torch.from_numpy(q).to(DEV))
            assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
            assert np.array_equal(_bits(emb), want)
            # packed gather is a verbatim copy of the stored rows
            pick = torch.tensor([0, 5, N - 1, 5], dtype=torch.int32, device=DEV)
            assert torch.equal(t.gather_packed(pick), t.storage[pick.long()])
    finally:
        if created:
            dist.destroy_process_group()


def test_offloaded_tier_zero_copy_and_staged():
    """Pinned-host table: zero-copy through the fused kernel, and the staged (host gather + async copy) variant."""
    sb, S = _mods()
    from scone_b200.offload import StagedHostLookup
    N, D, V, max_n, B, L = 6000, 1024, 400, 5, 8, 300
    toks, lens = S.make_vocab_numpy(N, max_n, V, seed=51)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=52)
    rows = S.make_rows_numpy(N, D, seed=53)
    base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=54), "bf16")
    want, wid, wlen = po.embed_forward(vocab_dict(toks, lens), max_n, po.OracleTable.from_fp32(rows, "int8"), base_bits, q, "bf16")
    ix = _index(toks, lens)
    host = sb.CacheTable(N, D, "int8", tier="host")
    host.store(torch.from_numpy(rows).to(DEV))
    torch.cuda.synchronize()
    base = _from_bits(base_bits, torch.bfloat16)
    out, fid, ml = sb.embed_forward(ix, host, base, torch.from_numpy(q).to(DEV))
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(_bits(out), want)
    for m in (1, 3, 4):
        st = StagedHostLookup(ix, host, base, micro_batches=m, max_positions=B * L, threads=4)
        out2, fid2, ml2 = st.lookup(torch.from_numpy(q).to(DEV))
        torch.cuda.synchronize()
        assert np.array_equal(fid2.cpu().numpy(), wid) and np.array_equal(ml2.cpu().numpy(), wlen)
        assert np.array_equal(_bits(out2), want)


# ---- SURVEY 8f "next" rows -------------------------------------------------------------------------------------------

def test_fit_device_matches_reference_fit():
    sb, _ = _mods()
    for name in ("fit_small.npz", "fit_medium.npz"):       # fit_medium: the max_f_grams cut falls inside a run of equal counts
        z = load_golden(name)
        offs = z["corpus_offs"]
        corpus = [z["corpus_flat"][offs[i]:offs[i + 1]].tolist() for i in range(len(offs) - 1)]
        ex = sb.NGramExtractor(int(z["max_n"]), int(z["min_freq"]), int(z["max_f_grams"])).fit_device(corpus, verbose=False)
        t, l = ex.vocab_arrays()
        assert np.array_equal(t, z["vocab_tokens"]) and np.array_equal(l, z["vocab_lens"]), name
    ex = sb.NGramExtractor(3, 1, 100).fit_device([[1, 2, 3, 4, 1, 2, 3], [2, 3, 4, 5], [1, 2, 9]], verbose=False)
    assert np.array_equal(ex.vocab_arrays()[0], load_golden("kat0.npz")["vocab_tokens"])
    assert sb.NGramExtractor(2, 2, 3).fit_device([[7, 8, 7, 8, 9]], verbose=False).f_gram_to_id == {(7,): 0, (8,): 1, (7, 8): 2}
    rng = np.random.default_rng(12)
    for _ in range(15):
        corpus = [rng.integers(0, 15, size=int(rng.integers(0, 40))).tolist() for _ in range(int(rng.integers(1, 9)))]
        max_n, min_freq, cap = int(rng.integers(1, 6)), int(rng.integers(1, 4)), int(rng.integers(1, 80))
        a = sb.NGramExtractor(max_n, min_freq, cap).fit_device(corpus, verbose=False)
        want = po.fit(corpus, max_n, min_freq, cap)
        assert [a.id_to_f_gram[i] for i in range(len(a))] == want
    # a corpus of 2 M tokens: identical to the host fit (which is pinned to the reference), many ties, truncation at work
    big = [rng.integers(0, 3000, size=int(rng.integers(10, 4000))).tolist() for _ in range(1000)]
    h = sb.NGramExtractor(4, 3, 200_000).fit(big, verbose=False)
    d = sb.NGramExtractor(4, 3, 200_000).fit_device(big, verbose=False)
    assert np.array_equal(h.vocab_arrays()[0], d.vocab_arrays()[0]) and np.array_equal(h.vocab_arrays()[1], d.vocab_arrays()[1])
    assert len(d) > 10_000
    with pytest.raises(ValueError):
        sb.NGramExtractor(2, 1, 10).fit_device([[3, -1, 3]], verbose=False)


def test_binary_format_and_reference_memmap_import(tmp_path):
    sb, S = _mods()
    z = load_golden("cache_small.npz")
    ex = sb.NGramExtractor.from_arrays(z["vocab_tokens"], z["vocab_lens"])
    N, D = z["rows"].shape
    for quant in ("fp16", "int4" if D % 128 == 0 else "int8"):
        cache = sb.EmbeddingCache(ex, D, quant=quant)
        cache.cache_embeddings(list(range(0, N, 2)), torch.from_numpy(z["rows"][0::2]), verbose=False)
        p = str(tmp_path / f"cache_{quant}.bin")
        cache.save_binary(p)
        back = sb.EmbeddingCache.load_binary(p, ex)
        assert back.quant == quant and torch.equal(back.table.storage, cache.table.storage)
        assert len(back.embeddings) == len(range(0, N, 2)) and 1 not in back.embeddings and 2 in back.embeddings
        host = sb.EmbeddingCache.load_binary(p, ex, cache_dir=str(tmp_path), use_memory_map=True)
        assert host.tier == "host" and torch.equal(host.table.storage, cache.table.storage.cpu())
    # the raw fp32 file the reference's memmap backend leaves behind (embedding_cache.py:84-91)
    raw = str(tmp_path / "embeddings.npy")
    mm = np.memmap(raw, dtype=np.float32, mode="w+", shape=(N, D))
    mm[:] = z["rows"]
    mm.flush()
    imp = sb.EmbeddingCache.from_reference_memmap(raw, ex, D)
    assert np.array_equal(imp.get_embeddings(z["pick"].tolist()).numpy().view(np.uint32), z["gathered"].view(np.uint32))


def test_reference_code_mean_mode_golden():
    """engine.py:235-259 re-enacted on the reference objects (golden `assembled`) vs the optional mean mode."""
    sb, _ = _mods()
    z = load_golden("cache_small.npz")
    ex = sb.NGramExtractor.from_arrays(z["vocab_tokens"], z["vocab_lens"])
    N, D = z["rows"].shape
    q = torch.from_numpy(z["query"])[None].to(DEV)
    # default storage (fp32 rows, as in the reference): the engine's tensor bit for bit
    c32 = sb.EmbeddingCache(ex, D)
    c32.cache_embeddings(list(range(N)), torch.from_numpy(z["rows"]), verbose=False)
    got32 = c32.assemble_mean(q)[0].cpu().numpy()
    assert np.array_equal(got32.view(np.uint32), z["assembled"].view(np.uint32))
    cache = sb.EmbeddingCache(ex, D, quant="fp16")
    cache.cache_embeddings(list(range(N)), torch.from_numpy(z["rows"]), verbose=False)
    got = cache.assemble_mean(q)[0].cpu().numpy()
    # exact against the oracle's restatement over the rows as stored (fp16), close to the reference's fp32 rows
    stored = z["rows"].astype(np.float16).astype(np.float32)
    want = po.assemble_mean(vocab_dict(z["vocab_tokens"], z["vocab_lens"]), int(z["max_n"]), lambda ids: stored[ids],
                            z["query"].tolist(), D)
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-9)
    np.testing.assert_allclose(got, z["assembled"], rtol=0, atol=2e-5)
    assert np.array_equal(got == 0, z["assembled"] == 0)              # zeros exactly where the reference has none
    # batched, other formats: against the oracle on dequantised rows
    from scone_b200.utils import synthetic as S
    toks, lens = S.make_vocab_numpy(1500, 5, 120, seed=61, min_n=1)
    rows = S.make_rows_numpy(1500, 256, seed=62)
    qq = S.make_stream_numpy(toks, lens, 3, 90, 120, seed=63)
    for quant in ("int8", "int4"):
        tab = po.OracleTable.from_fp32(rows, quant)
        ix = _index(toks, lens)
        t = sb.CacheTable(1500, 256, quant)
        t.store(torch.from_numpy(rows).to(DEV))
        g = sb.embed_mean_forward(ix, t, torch.from_numpy(qq).to(DEV)).cpu().numpy()
        g2i = vocab_dict(toks, lens)
        for b in range(3):
            w = po.assemble_mean(g2i, 5, tab.rows_fp32, qq[b].tolist(), 256)
            np.testing.assert_allclose(g[b], w, rtol=0, atol=1e-8)


@pytest.mark.parametrize("quant", ["fp32", "fp16", "int8", "int4"])
def test_mean_mode_16bit_outputs_are_the_rounded_fp32_output(quant):
    """The mean kernel computes each fp32 mean once and rounds it to the output type: its bf16 / fp16 outputs are bit for bit
    the round-to-nearest-even cast of its fp32 output on the same inputs, for every stored format."""
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(1500, 5, 120, seed=71, min_n=1)
    rows = S.make_rows_numpy(1500, 264, seed=72)                 # 33 chunks: one lane takes two
    qq = torch.from_numpy(S.make_stream_numpy(toks, lens, 3, 90, 120, seed=73)).to(DEV)
    ix = _index(toks, lens)
    t = sb.CacheTable(1500, 264, quant, group=8 if quant == "int4" else 128)
    t.store(torch.from_numpy(rows).to(DEV))
    g32 = sb.embed_mean_forward(ix, t, qq).cpu().numpy()
    assert np.count_nonzero(g32) > g32.size // 2
    for name, dt in TORCH_DT.items():
        g16 = _bits(sb.embed_mean_forward(ix, t, qq, dtype=dt))
        assert np.array_equal(g16, po.cast_bits(g32, name)), name


def test_host_pipeline_matches_direct_call():
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(3000, 4, 300, seed=71)
    ix = _index(toks, lens)
    t = sb.CacheTable(3000, 256, "int8")
    t.store(torch.from_numpy(S.make_rows_numpy(3000, 256, seed=72)).to(DEV))
    base = torch.from_numpy(S.make_rows_numpy(300, 256, seed=73)).to(DEV).to(torch.bfloat16)
    B, L = 4, 160
    hb = [torch.from_numpy(S.make_stream_numpy(toks, lens, B, L, 300, seed=80 + k)).pin_memory() for k in range(7)]
    pipe = sb.HostPipeline(ix, t, base, (B, L))
    ex = sb.NGramExtractor.from_arrays(toks, lens)
    cache = sb.EmbeddingCache(ex, 256, quant="int8")
    cache.cache_embeddings(list(range(3000)), torch.from_numpy(S.make_rows_numpy(3000, 256, seed=72)), verbose=False)
    cache.set_base_embedding(base)
    pipe2 = cache.host_pipeline((B, L))
    r = [pipe2.submit(h) for h in hb[:3]][-1]                    # 4 slots: the first result comes back on the third submit
    assert torch.equal(r[0], sb.embed_forward(ix, t, base, hb[0].to(DEV))[0])
    pipe2.flush()
    got = []
    for h in hb:
        r = pipe.submit(h)
        if r is not None:
            got.append((r[0].clone(), r[1].clone(), r[2].clone()))
    got += [(r[0].clone(), r[1].clone(), r[2].clone()) for r in pipe.flush()]
    assert len(got) == len(hb)
    for h, (e, i, l) in zip(hb, got):
        we, wi, wl = sb.embed_forward(ix, t, base, h.to(DEV))
        assert torch.equal(e, we) and torch.equal(i.to(DEV), wi) and torch.equal(l.to(DEV), wl)


def test_hypothesis_gpu_lookup_vs_oracle():
    from hypothesis import given, settings, strategies as st

    @settings(max_examples=40, deadline=None)
    @given(st.data())
    def run(data):
        max_n = data.draw(st.integers(1, 7))
        V = data.draw(st.integers(1, 10))
        grams = data.draw(st.lists(st.lists(st.integers(0, V - 1), min_size=1, max_size=max_n).map(tuple), max_size=60, unique=True))
        B = data.draw(st.integers(1, 3))
        L = data.draw(st.integers(1, 70))
        q = np.array(data.draw(st.lists(st.lists(st.integers(0, V), min_size=L, max_size=L), min_size=B, max_size=B)), dtype=np.int64)
        toks = np.full((len(grams), max_n), -1, np.int32)
        lens = np.zeros(len(grams), np.uint8)
        for i, g in enumerate(grams):
            toks[i, :len(g)] = g
            lens[i] = len(g)
        ix = _index(toks, lens, load_factor=data.draw(st.sampled_from([0.1, 0.25, 0.5, 0.9])))
        fid, ml = ix.lookup(torch.from_numpy(q).to(DEV))
        wid, wl = po.match_batch({g: i for i, g in enumerate(grams)}, max_n, q)
        assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wl)
        ix.close()

    run()


@pytest.mark.parametrize("quant,D,max_n", [("fp16", 8192, 5), ("int8", 16384, 3), ("int4", 16384, 2), ("fp16", 4096, 1)])
def test_embed_forward_rows_too_wide_for_the_ring(quant, D, max_n):
    """Rows that do not fit the shared-memory ring take the register-load variant of the kernel."""
    _embed_case(quant, "bf16", D, max_n, N=60 if max_n == 1 else 600, V=300, B=2, L=75, seed=D + max_n, min_n=1 if max_n < 3 else 2)


def test_embed_forward_all_hits_and_all_misses():
    sb, S = _mods()
    toks = np.array([[5, -1], [5, 5]], np.int32)
    lens = np.array([1, 2], np.uint8)
    ix = _index(toks, lens)
    t = sb.CacheTable(2, 256, "int8")
    rows = S.make_rows_numpy(2, 256, seed=1)
    t.store(torch.from_numpy(rows).to(DEV))
    base = torch.from_numpy(S.make_rows_numpy(10, 256, seed=2)).to(DEV).to(torch.bfloat16)
    allhit = torch.full((3, 40), 5, dtype=torch.long, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, allhit)
    assert fid[:, 0].tolist() == [0, 0, 0] and bool((fid[:, 1:] == 1).all()) and bool((ml[:, 1:] == 2).all())
    assert torch.equal(out[:, 1:], t.gather(torch.tensor([1], device=DEV), torch.bfloat16).expand(3, 39, 256))
    allmiss = torch.full((3, 40), 7, dtype=torch.long, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, allmiss)
    assert bool((fid == -1).all()) and bool((ml == 0).all()) and torch.equal(out, base[7].expand(3, 40, 256))


def test_cuda_graph_replay_and_pdl_give_identical_results(monkeypatch):
    """The hot call is asynchronous and capture-safe: K launches replayed from one CUDA graph (as bench.py times them)
    reproduce the eager results bit for bit (every launch uses programmatic dependent launch)."""
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(4000, 4, 500, seed=91)
    ix = _index(toks, lens)
    t = sb.CacheTable(4000, 1024, "int8")
    t.store(torch.from_numpy(S.make_rows_numpy(4000, 1024, seed=92)).to(DEV))
    base = torch.from_numpy(S.make_rows_numpy(500, 1024, seed=93)).to(DEV).to(torch.bfloat16)
    qs = [torch.from_numpy(S.make_stream_numpy(toks, lens, 6, 500, 500, seed=94 + k)).to(DEV) for k in range(3)]
    eager = [sb.embed_forward(ix, t, base, q) for q in qs]
    outs = [torch.empty_like(e[0]) for e in eager]
    ids = [torch.empty_like(e[1]) for e in eager]
    lens_o = [torch.empty_like(e[2]) for e in eager]
    for _ in range(2):
        stream = torch.cuda.Stream()
        with torch.cuda.stream(stream):
            for k, q in enumerate(qs):
                sb.embed_forward(ix, t, base, q, out=outs[k], out_id=ids[k], out_len=lens_o[k])
            stream.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=stream):
                for rep in range(2):
                    for k, q in enumerate(qs):
                        sb.embed_forward(ix, t, base, q, out=outs[k], out_id=ids[k], out_len=lens_o[k])
            for o in outs:
                o.zero_()
            g.replay()
            stream.synchronize()
        for k in range(3):
            assert torch.equal(outs[k], eager[k][0]) and torch.equal(ids[k], eager[k][1]) and torch.equal(lens_o[k], eager[k][2])


def test_reads_cache_file_written_by_the_reference():
    """tests/golden/ref_cache.npy was written by the unmodified reference's EmbeddingCache.save (dict backend, every third id)."""
    import os
    from conftest import GOLDEN
    sb, _ = _mods()
    z = load_golden("cache_small.npz")
    ex = sb.NGramExtractor.load(os.path.join(GOLDEN, "ref_extractor.npy"))
    cache = sb.EmbeddingCache.load(os.path.join(GOLDEN, "ref_cache.npy"), ex)
    N = z["rows"].shape[0]
    keep = list(range(0, N, 3))
    assert len(cache.embeddings) == len(keep) and 0 in cache.embeddings and 1 not in cache.embeddings
    got = cache.get_embeddings(keep)
    assert torch.equal(got, torch.from_numpy(z["rows"][keep]))           # fp32 rows in, the same fp32 rows out
    with pytest.raises(KeyError):
        cache.get_embeddings([1])
    # the fused path refuses a table with holes, like the reference's KeyError for a matched f-gram without a row
    cache.set_base_embedding(torch.zeros(64, z["rows"].shape[1]))
    q = torch.from_numpy(z["query"])[None].to(DEV)
    with pytest.raises(KeyError):
        cache.lookup(q)
    out, fid, _ = cache.lookup(q, strict=False)                          # opt-out: uncached rows read as zeros
    assert np.array_equal(fid.cpu().numpy()[0], z["fgram_id"])


def test_inputs_stable_flag_never_changes_a_result():
    """SCONE_EMBED_INPUTS_STABLE only moves the point where the kernel waits for its predecessor (matching and row fetches
    start under the previous launch's tail); eager, back to back, and replayed from a CUDA graph the results stay bit-identical
    to the default launches -- for the plain path, the fused position add and the additive combine."""
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(6000, 4, 500, seed=101)
    ix = _index(toks, lens)
    for quant, D in (("int8", 1024), ("int4", 4096), ("fp32", 768)):
        t = sb.CacheTable(6000, D, quant)
        t.store(torch.from_numpy(S.make_rows_numpy(6000, D, seed=102)).to(DEV))
        base = torch.from_numpy(S.make_rows_numpy(500, D, seed=103)).to(DEV).to(torch.bfloat16)
        pos = torch.from_numpy(S.make_rows_numpy(640, D, seed=104)).to(DEV).to(torch.bfloat16)
        qs = [torch.from_numpy(S.make_stream_numpy(toks, lens, 8, 640, 500, seed=105 + k)).to(DEV) for k in range(4)]
        for kw in ({}, {"pos_emb": pos}, {"combine": "add"}):
            want = [sb.embed_forward(ix, t, base, q, **kw) for q in qs]
            torch.cuda.synchronize()
            outs = [torch.zeros_like(w[0]) for w in want]
            ids = [torch.zeros_like(w[1]) for w in want]
            lns = [torch.zeros_like(w[2]) for w in want]
            stream = torch.cuda.Stream()
            with torch.cuda.stream(stream):
                for rep in range(3):                       # eager, back to back: launch k+1 starts under launch k
                    for k, q in enumerate(qs):
                        sb.embed_forward(ix, t, base, q, out=outs[k], out_id=ids[k], out_len=lns[k], inputs_stable=True, **kw)
                stream.synchronize()
                for k in range(4):
                    assert torch.equal(outs[k], want[k][0]) and torch.equal(ids[k], want[k][1]) and torch.equal(lns[k], want[k][2])
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=stream):
                    for rep in range(3):
                        for k, q in enumerate(qs):
                            sb.embed_forward(ix, t, base, q, out=outs[k], out_id=ids[k], out_len=lns[k], inputs_stable=True, **kw)
                for o in outs:
                    o.zero_()
                g.replay()
                g.replay()
                stream.synchronize()
            for k in range(4):
                assert torch.equal(outs[k], want[k][0]) and torch.equal(ids[k], want[k][1]) and torch.equal(lns[k], want[k][2])


def test_every_fused_entry_validates_its_buffers():
    """A short / mistyped pos_emb or a mis-shaped out must be a ValueError, not an out-of-bounds bulk copy -- also on the
    resolved-ids gather and on the sharded entry (world 1 here)."""
    sb, S = _mods()
    toks, lens = S.make_vocab_numpy(300, 3, 80, seed=111)
    ix = _index(toks, lens)
    t = sb.CacheTable(300, 64, "fp16")
    base = torch.zeros(80, 64, device=DEV, dtype=torch.bfloat16)
    q = torch.from_numpy(S.make_stream_numpy(toks, lens, 2, 50, 80, seed=112)).to(DEV)
    fid, _ = ix.lookup(q)
    for bad in (dict(pos_emb=torch.zeros(10, 64, device=DEV, dtype=torch.bfloat16)),          # shorter than L
                dict(pos_emb=torch.zeros(50, 64, device=DEV, dtype=torch.float32)),           # wrong dtype
                dict(out=torch.zeros(2, 50, 32, device=DEV, dtype=torch.bfloat16)),           # wrong shape
                dict(out=torch.zeros(2, 50, 64, device=DEV, dtype=torch.float16))):           # wrong dtype
        with pytest.raises(ValueError):
            sb.embed_forward(ix, t, base, q, **bad)
        with pytest.raises(ValueError):
            sb.embed_gather(t, base, q, fid, **bad)
    with pytest.raises(ValueError):
        sb.embed_gather(t, base.float(), q, fid)
    with pytest.raises(ValueError):
        sb.embed_gather(t, base[:, :32].contiguous(), q, fid)
    with pytest.raises(ValueError):
        sb.embed_forward(ix, t, base, q, out_id=torch.zeros(2, 50, device=DEV, dtype=torch.int64))


def test_config3_full_size_against_c_oracle(index_format):
    """BASELINE config 3 at its named size on the device: 10 M f-grams (V = 128 000: compact 20-bit-token slots, a 20 MB
    pre-filter; and once more with 32-byte slots -- 1.28 GB addressed past 2^31 bytes -- and no filter), D = 4096 INT4 g128
    rows (21 GB table), 256 x 2048 positions.  f-gram ids and match lengths of the WHOLE batch and the embeddings of 8 batch rows against the C oracle
    (built over the whole vocabulary; the table is one quantised 65 536-row block tiled, which is how bench.py fills it),
    plus the oracle-independent properties of the whole output."""
    if index_format != "auto":
        pytest.skip("one pass at this size: the 10 M-f-gram vocabulary takes the 32-byte slot format and no filter by itself")
    sb, S = _mods()
    N, D, V, max_n, B, L, BLK = 10_000_000, 4096, 128_000, 5, 256, 2048, 65536
    toks, lens, longest = S.make_vocab_device(N, max_n, V, seed=0, device=DEV, return_longest=True)
    ix = sb.FGramIndex(toks, lens)
    assert ix.slot_format == "compact20" and ix.slot_bytes == 16 and ix.filter_bytes == 20_000_000 and ix.bytes > (600 << 20)
    blk = sb.CacheTable(BLK, D, "int4")
    S.fill_table_device(blk, seed=2)
    t = sb.CacheTable(N, D, "int4")
    for s0 in range(0, N, BLK):
        k = min(BLK, N - s0)
        t.storage[s0:s0 + k].copy_(blk.storage[:k])
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device=DEV)
    q = S.make_stream_device(toks, lens, B, L, V, seed=100, p_plant=1.0, pick_ids=longest)
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    out, fid, ml = sb.embed_forward(ix, t, base, q, status=status)
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    # (1) the match result of all 524 288 positions against the C oracle
    cix = COracleIndex(toks.cpu().numpy(), lens.cpu().numpy())
    q_h = q.cpu().numpy()
    wid, wlen = cix.match(q_h, nthreads=16)
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    assert 0.7 < (wid >= 0).mean() < 0.9 and int(wid.max()) > (1 << 23)          # rows beyond 2^31 bytes of table are touched
    # (2) embeddings of 8 batch rows, bit for bit: oracle dequant of the tiled block's row (id % BLK), fallback rows elsewhere
    blk_h = blk.storage.cpu().numpy()
    tab = po.OracleTable("int4", D, blk_h[:, :D // 2], blk_h[:, t.scale_offset:t.scale_offset + 2 * (D // 128)].copy().view(np.float16))
    base_h = _bits(base)
    for b in (0, 1, 2, 3, 100, 101, 254, 255):
        w_, h_ = wid[b], wid[b] >= 0
        want = np.empty((L, D), np.uint16)
        want[~h_] = base_h[q_h[b][~h_]]
        want[h_] = po.cast_bits(tab.rows_fp32(w_[h_].astype(np.int64) % BLK), "bf16")
        assert np.array_equal(_bits(out[b]), want), b
    # (3) oracle-independent properties over the whole output
    miss = fid < 0
    assert torch.equal(out[miss], base[q[miss]])                                      # misses are the fallback rows
    sel = torch.nonzero(fid.flatten() >= 0).flatten()[:: 997]
    assert torch.equal(out.flatten(0, 1)[sel], t.gather(fid.flatten()[sel].long(), torch.bfloat16))   # hits equal table.gather
    i = torch.nonzero(ml.flatten() == 5).flatten()[:: 1009]                             # matched tokens are the window's suffix
    win = torch.stack([q.flatten()[i - 4 + k] for k in range(5)], dim=1).to(torch.int32)
    assert torch.equal(win, toks[fid.flatten()[i].long()])
    out2, fid2, _ = sb.embed_forward(ix, t, base, q, inputs_stable=True)
    assert torch.equal(out2, out) and torch.equal(fid2, fid)                          # deterministic
    # (4) the same vocabulary in 32-byte slots without a filter (slot addresses beyond 2^31 bytes), and through the single-ring kernel
    import os
    os.environ.update(SCONE_INDEX_FORMAT="wide", SCONE_INDEX_FILTER="never", SCONE_EMBED_PIPE="0")
    try:
        ixw = sb.FGramIndex(toks, lens)
        assert ixw.slot_bytes == 32 and ixw.filter_bytes == 0 and ixw.bytes > (1 << 30)
        out3, fid3, ml3 = sb.embed_forward(ixw, t, base, q)
        assert torch.equal(fid3, fid) and torch.equal(ml3, ml) and torch.equal(out3, out)
    finally:
        for k_ in ("SCONE_INDEX_FORMAT", "SCONE_INDEX_FILTER", "SCONE_EMBED_PIPE"):
            os.environ.pop(k_, None)


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_tier_two_gpus_reference_api(tmp_path):
    """The row-sharded tier on 2 GPUs (torchrun, NCCL): lookup through both exchange variants and the reference-API methods
    (get_embeddings, embeddings[...], get_token_embeddings) with GLOBAL ids, against the C oracle on the unsharded table."""
    import os
    import subprocess
    import sys
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29571", os.path.join(ROOT, "tests", "multi_gpu", "run_sharded.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "MISMATCH" not in p.stdout and p.stdout.count("OK") >= 8


@pytest.mark.parametrize("Hf,H,k", [(384, 768, 1000), (768, 1024, 517), (96, 256, 300), (1024, 4096, 260), (8, 64, 1), (72, 320, 129),
                                    (40, 448, 257), (64, 2048, 9000), (48, 1280, 7000), (32, 512, 40000)])
def test_projection_fold(Hf, H, k):
    """table[row] = quantise(rows @ W^T): the reference's bias-free f_gram_projection (language_model.py:172-176, :236) folded
    into the table build by a tcgen05 / TMEM GEMM whose epilogue is the quantiser.
    (1) the unquantised result against the exact product of the bf16-rounded inputs, within the accumulation-order bound of
        oracle/py_oracle.py::fold_projection;
    (2) every quantised format bit-identical to scone_table_store (the oracle-pinned quantiser) applied to (1): the epilogue IS
        that quantiser;
    (3) so the dequantised rows are within half a quantisation step (+ the bound) of the exact product."""
    sb, S = _mods()
    rng = np.random.default_rng(Hf + H)
    rows = (rng.standard_normal((k, Hf)) * 0.5).astype(np.float32)
    W = (rng.standard_normal((H, Hf)) * (1.0 / np.sqrt(Hf))).astype(np.float32)
    rows[min(3, k - 1)] = 0.0                       # an all-zero row: scale 1
    P, bound = po.fold_projection(rows, W)
    perm = rng.permutation(k)
    import os
    # both tensor-core paths: CTA pairs on one 256 x 256 tile (tcgen05.mma.cta_group::2; the default for FP16 tables with
    # K >= 512) and one 128 x 256 tile per CTA
    xs = {}
    for two_sm in ("0", "1"):
        os.environ["SCONE_FOLD_2SM"] = two_sm
        try:
            t32 = sb.CacheTable(k, H, "fp32")
            t32.store_projected(torch.from_numpy(rows).to(DEV), torch.from_numpy(W).to(DEV), row_ids=torch.from_numpy(perm).to(DEV))
        finally:
            os.environ.pop("SCONE_FOLD_2SM", None)
        x = t32.gather(torch.arange(k, device=DEV)).cpu().numpy()
        xs[two_sm] = x
        x_src = x[perm]                             # row r of the input went to table row perm[r]
        assert np.all(np.abs(x_src - P) <= bound + 1e-30), (two_sm, float(np.max(np.abs(x_src - P) - bound)))
        assert np.array_equal(x_src[min(3, k - 1)], np.zeros(H, np.float32))
    # INT8 twice: row absmax exchanged between the CTAs of a cluster (one sweep; the default for 256 < H <= 2048; the large-k
    # shapes give every cluster several row tiles) and the two-sweep path
    for quant in ("fp16", "fp16-pair-tile", "int8", "int8-two-sweeps", "int8-two-sweeps-pair-tile", "int4", "int4-pair-tile", "int4-g32",
                  "int4-g64-pair-tile"):
        group = int(quant.split("-g")[1].split("-")[0]) if "-g" in quant else 128
        if quant.startswith("int4") and H % group:
            continue                                # INT4 groups of `group` columns
        if "two-sweeps" in quant:
            os.environ["SCONE_FOLD_XCH"] = "0"
        two_sm = "1" if quant.endswith("pair-tile") else "0"
        os.environ["SCONE_FOLD_2SM"] = two_sm
        x = xs[two_sm]                              # the fp32 product of the same tensor-core path
        quant = quant.split("-")[0]
        tq = sb.CacheTable(k, H, quant, group=group)
        try:
            tq.store_projected(torch.from_numpy(rows).to(DEV), torch.from_numpy(W).to(DEV), row_ids=torch.from_numpy(perm).to(DEV))
        finally:
            os.environ.pop("SCONE_FOLD_XCH", None)
            os.environ.pop("SCONE_FOLD_2SM", None)
        ref = sb.CacheTable(k, H, quant, group=group)
        ref.store(torch.from_numpy(x).to(DEV))
        assert torch.equal(tq.storage, ref.storage), quant
        dq = tq.gather(torch.arange(k, device=DEV)).cpu().numpy()[perm]
        if quant == "fp16":
            step = np.maximum(np.abs(P) * 2.0 ** -10, 2.0 ** -24)
        elif quant == "int8":
            step = (np.abs(P).max(axis=1, keepdims=True) / 127.0) * np.ones_like(P)
        else:
            step = np.repeat((np.abs(P).reshape(k, H // group, group).max(axis=2) / 7.0).astype(np.float16).astype(np.float32), group, axis=1)
        assert np.all(np.abs(dq - P) <= 0.51 * step + 4 * bound + 1e-30), (quant, group)
    # the epilogue's per-group loop takes 32, 64 or 128 columns
    for group in (16, 256):
        if H % group == 0:
            with pytest.raises(ValueError, match="group"):
                sb.CacheTable(k, H, "int4", group=group).store_projected(torch.from_numpy(rows).to(DEV), torch.from_numpy(W).to(DEV))
    # the drop-in entry: cache_embeddings(..., projection=W) then lookup serves the projected rows
    if k < 200:
        return
    toks, lens = S.make_vocab_numpy(k, 3, 200, seed=5)
    ex = sb.NGramExtractor.from_arrays(toks, lens)
    cache = sb.EmbeddingCache(ex, H, quant="fp16", out_dtype=torch.float16)
    cache.cache_embeddings(list(range(k)), torch.from_numpy(rows), verbose=False, projection=torch.from_numpy(W))
    got = cache.get_embeddings(list(range(k))).numpy()
    ref16 = sb.CacheTable(k, H, "fp16")
    t_id = sb.CacheTable(k, H, "fp32")
    t_id.store_projected(torch.from_numpy(rows).to(DEV), torch.from_numpy(W).to(DEV))
    ref16.store(t_id.gather(torch.arange(k, device=DEV)))
    assert np.array_equal(got, ref16.gather(torch.arange(k, device=DEV)).cpu().numpy())
    with pytest.raises(ValueError):
        cache.cache_embeddings([0], torch.zeros(1, Hf), projection=torch.zeros(H + 64, Hf))
