"""CPU tests of the host side: C-ABI surface, drop-in host logic, synthetic generators."""

import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden
from oracle import py_oracle as po


def test_library_loads_and_exports_every_declared_symbol():
    from scone_b200 import _lib, build
    build.build()
    L = _lib.load()
    header = open(os.path.join(ROOT, "include", "scone_b200.h")).read()
    declared = set(re.findall(r"\b(scone_[a-z0-9_]+)\s*\(", header))
    declared -= {"scone_index_create_ex"}
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert getattr(L, name) is not None
    assert L.scone_version() == _lib.ABI_VERSION == int(re.search(r"#define SCONE_B200_VERSION (\d+)", header).group(1))
    assert ctypes.sizeof(_lib.TableDesc) == 40 and ctypes.sizeof(_lib.IndexInfo) == 56 and ctypes.sizeof(_lib.EmbedOpts) == 16


def test_table_layout_matches_oracle_packing():
    from scone_b200 import table_layout
    from scone_b200.utils.synthetic import pack_table_numpy
    rows = (np.random.default_rng(0).standard_normal((4, 1024)) * 0.02).astype(np.float32)
    for quant, want in (("fp32", (4096, 0)), ("fp16", (2048, 0)), ("int8", (1056, 1024)), ("int4", (544, 512))):
        assert table_layout(quant, 1024) == want
        t = po.OracleTable.from_fp32(rows, quant)
        _, stride, soff = pack_table_numpy(quant, t.payload, t.scales)
        assert (stride, soff) == want
    assert table_layout("int4", 4096) == (2112, 2048)            # SURVEY 8d: R = D/2 + 2 D/128
    with pytest.raises(ValueError):
        table_layout("int4", 100)
    with pytest.raises(ValueError):
        table_layout("fp16", 12)


def test_invalid_arguments_fail_loudly_without_a_gpu():
    import torch
    import scone_b200
    with pytest.raises(ValueError):
        scone_b200.FGramIndex(torch.zeros((1, 2), dtype=torch.int32), torch.ones((1,), dtype=torch.uint8))   # CPU tensors
    if not torch.cuda.is_available():
        ex = scone_b200.NGramExtractor.from_arrays(np.array([[1, 2]], np.int32), np.array([2], np.uint8))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ex.get_token_f_grams([1, 2, 3])


def test_host_fit_matches_reference_fixtures():
    from scone_b200 import NGramExtractor
    for name in ("fit_small.npz", "fit_medium.npz"):       # fit_medium: the cut falls inside a run of equal counts
        z = load_golden(name)
        offs = z["corpus_offs"]
        corpus = [z["corpus_flat"][offs[i]:offs[i + 1]].tolist() for i in range(len(offs) - 1)]
        ex = NGramExtractor(int(z["max_n"]), int(z["min_freq"]), int(z["max_f_grams"])).fit(corpus, verbose=False)
        t, l = ex.vocab_arrays()
        assert np.array_equal(t, z["vocab_tokens"]) and np.array_equal(l, z["vocab_lens"]), name
    k = load_golden("kat0.npz")
    ex = NGramExtractor(3, 1, 100).fit([[1, 2, 3, 4, 1, 2, 3], [2, 3, 4, 5], [1, 2, 9]], verbose=False)
    assert np.array_equal(ex.vocab_arrays()[0], k["vocab_tokens"])
    ex = NGramExtractor(2, 2, 3).fit([[7, 8, 7, 8, 9]], verbose=False)
    assert ex.f_gram_to_id == {(7,): 0, (8,): 1, (7, 8): 2}
    with pytest.raises(ValueError):
        NGramExtractor(2, 1, 10).fit([[3, -1, 3, -1]], verbose=False)          # -1 is the arrays' padding value: refused, not miscounted
    # fuzz against the oracle's restatement of fit
    rng = np.random.default_rng(8)
    for _ in range(25):
        corpus = [rng.integers(0, 12, size=int(rng.integers(0, 30))).tolist() for _ in range(int(rng.integers(1, 8)))]
        max_n, min_freq, cap = int(rng.integers(1, 5)), int(rng.integers(1, 4)), int(rng.integers(1, 60))
        ex = NGramExtractor(max_n, min_freq, cap).fit(corpus, verbose=False)
        want = po.fit(corpus, max_n, min_freq, cap)
        assert [ex.id_to_f_gram[i] for i in range(len(ex))] == want
        assert ex.extract_all_n_grams(corpus[0]) == po.extract_all_n_grams(corpus[0], max_n)


def test_extractor_save_load_reference_format(tmp_path):
    from scone_b200 import NGramExtractor
    ex = NGramExtractor(3, 1, 50).fit([[1, 2, 3, 1, 2], [4, 5]], verbose=False)
    p = str(tmp_path / "e.npy")
    ex.save(p)
    raw = np.load(p, allow_pickle=True).item()
    assert set(raw) == {"max_n", "min_freq", "max_f_grams", "f_gram_to_id"} and "1,2" in raw["f_gram_to_id"]
    back = NGramExtractor.load(p)
    assert back.f_gram_to_id == ex.f_gram_to_id and back.id_to_f_gram == ex.id_to_f_gram and back.f_grams == ex.f_grams


def test_synthetic_generators():
    from scone_b200.utils import synthetic as S
    t, l = S.make_vocab_numpy(2000, 5, 300, seed=1)
    keys = {tuple(t[i, :l[i]]) for i in range(2000)}
    assert len(keys) == 2000 and l.min() >= 2 and l.max() == 5 and (t[np.arange(2000), l - 1] >= 0).all()
    q = S.make_stream_numpy(t, l, 4, 128, 300, seed=2)
    assert q.shape == (4, 128) and q.min() >= 0 and q.max() < 300
    from conftest import vocab_dict
    fid, _ = po.match_batch(vocab_dict(t, l), 5, q)
    assert (fid >= 0).mean() > 0.5
    import torch
    td, ld, longest = S.make_vocab_device(5000, 4, 100, seed=0, device="cpu", return_longest=True)
    keys = {tuple(td[i, :ld[i]].tolist()) for i in range(5000)}
    assert len(keys) == 5000 and int(ld.min()) == 2 and int(ld.max()) == 4 and bool((ld[longest] == 4).all())
    qd = S.make_stream_device(td, ld, 2, 64, 100, seed=1, p_plant=1.0, pick_ids=longest)
    assert qd.shape == (2, 64) and qd.dtype == torch.int64
    fid, _ = po.match_batch(vocab_dict(td.numpy(), ld.numpy()), 4, qd.numpy())
    assert (fid >= 0).mean() > 0.7


def test_tiers_and_pipeline_refuse_cpu():
    """No CPU path anywhere: the tier / pipeline wrappers raise before touching the library when there is no CUDA tensor."""
    import torch
    import scone_b200 as sb
    from scone_b200 import sharded
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    with pytest.raises((ValueError, RuntimeError)):
        sb.CacheTable(4, 64, "int8")
    with pytest.raises(ValueError):
        sb.EmbeddingCache(sb.NGramExtractor.from_arrays(np.array([[1, 2]], np.int32), np.array([2], np.uint8)), 64, tier="nvme")
    assert sharded.shard_rows(10, 3, 4) == 2 and sharded.shard_rows(2, 3, 4) == 0


def _device_hash(tokens_reversed: np.ndarray, n: int) -> np.ndarray:
    """numpy mirror of hash_seed / hash_roll / hash_finish in scone_b200/csrc/common.cuh (uint64 arithmetic wraps)."""
    u = np.uint64
    h = np.full(tokens_reversed.shape[0], 0x243F6A8885A308D3, dtype=np.uint64)
    for k in range(n):
        h = (h ^ tokens_reversed[:, k].astype(np.uint64)) * u(0x9E3779B97F4A7C15)
        h ^= h >> u(29)
    h ^= u((n * 0xD6E8FEB86659FD93) & 0xFFFFFFFFFFFFFFFF)
    h ^= h >> u(33)
    h *= u(0xFF51AFD7ED558CCD)
    h ^= h >> u(33)
    h *= u(0xC4CEB9FE1A85EC53)
    h ^= h >> u(33)
    return h


@pytest.mark.parametrize("n_keys", [50_000, 300_000, 1_000_000])
def test_prefilter_parameters_give_the_documented_false_positive_rate(n_keys):
    """The index's Bloom pre-filter (index_format.cuh: filter_bits / filter_pass, index_plan.h: sizing) restated in numpy: 16+ bits per
    f-gram, two bits of one 32-bit word per key -> no false negatives, false positives of a few per cent at most (DESIGN.md
    section 3 quotes ~1.5 %).  Checks the design parameters; the CUDA code itself is held to the oracle by the GPU tests."""
    u = np.uint64
    rng = np.random.default_rng(n_keys)
    n = 4
    keys = rng.integers(0, 50_257, size=(n_keys, n), dtype=np.int64)
    probes = rng.integers(0, 50_257, size=(200_000, n), dtype=np.int64)
    words = max(1024, (n_keys + 1) // 2)                  # scone_index_create: 16 bits per key up to 12 M f-grams
    words = (words + 31) & ~31
    assert 16 * n_keys <= 32 * words < 16 * n_keys + 32 * 1024 + 1024
    def word_and_bits(h):
        w = ((h & u(0xFFFFFFFF)) * u(words)) >> u(32)     # index_format.cuh: filter_word
        b = (u(1) << ((h >> u(32)) & u(31))) | (u(1) << ((h >> u(37)) & u(31)))
        return w.astype(np.int64), b.astype(np.uint32)
    filt = np.zeros(words, dtype=np.uint32)
    w, b = word_and_bits(_device_hash(keys, n))
    np.bitwise_or.at(filt, w, b)
    assert ((filt[w] & b) == b).all()                      # no false negatives
    w2, b2 = word_and_bits(_device_hash(probes, n))
    passed = (filt[w2] & b2) == b2
    in_vocab = np.isin(probes.view([("", probes.dtype)] * n).ravel(), keys.view([("", keys.dtype)] * n).ravel())
    fp = (passed & ~in_vocab).sum() / max(1, (~in_vocab).sum())
    assert fp < 0.025, fp
    assert len(np.unique(_device_hash(keys, n))) > 0.999 * len(np.unique(keys, axis=0))     # the 64-bit hash itself does not collide


def test_combine_argument_is_validated_before_any_device_work():
    import scone_b200 as sb
    from scone_b200.table import embed_forward
    with pytest.raises(ValueError, match="combine"):
        embed_forward(None, None, None, torch.zeros((1, 4), dtype=torch.long), combine="mean")
    with pytest.raises(ValueError, match="combine"):
        sb.SconeInputEmbedding(None, torch.zeros(4, 8), combine="sum")


def test_header_cites_reference_for_every_entry_point():
    """include/scone_b200.h must say which reference code each compute entry point replaces (file:line)."""
    header = open(os.path.join(ROOT, "include", "scone_b200.h")).read()
    for needle in ("n_gram_extractor.py:121-122", "embedding_cache.py:173", "embedding_cache.py:113-147", "embedding_cache.py:56-111",
                   "engine.py:235-266", "language_model.py:239", "engine.py:235-259", "n_gram_extractor.py:106-126"):
        assert needle in header, needle
    integration = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    from scone_b200 import _lib
    for sym in _lib.SYMBOLS:
        if sym.startswith(("scone_index", "scone_table", "scone_embed", "scone_pipeline", "scone_host")):
            stem = sym if sym in integration else sym.rsplit("_", 1)[0]
            assert stem in integration, sym


def test_library_reads_only_the_path_overrides_the_gpu_tests_set():
    """The library reads five environment variables, each forcing a kernel, slot format, filter or fold path that is otherwise
    chosen from the inputs.  tests/test_gpu_parity.py sets every one of them to run each path; a renamed or added switch fails here."""
    overrides = {"SCONE_EMBED_PIPE", "SCONE_INDEX_FORMAT", "SCONE_INDEX_FILTER", "SCONE_FOLD_2SM", "SCONE_FOLD_XCH"}
    csrc = os.path.join(ROOT, "scone_b200", "csrc")
    read = set()
    for name in sorted(os.listdir(csrc)):
        src = open(os.path.join(csrc, name)).read()
        names = re.findall(r'getenv\(\s*"([^"]*)"\s*\)', src)
        assert len(names) == src.count("getenv("), f"{name}: getenv with a name that is not a string literal"
        read |= set(names)
    assert read == overrides
    parity = open(os.path.join(ROOT, "tests", "test_gpu_parity.py")).read()
    for var in sorted(overrides):
        assert re.search(rf'setenv\(\s*"{var}"|os\.environ\[\s*"{var}"\s*\]\s*=[^=]|\b{var}\s*=\s*"', parity), var


def test_host_gather_rows_is_pure_host_code():
    """scone_host_gather_rows (staged offload tier) runs without a GPU: multi-threaded row gather into a staging buffer."""
    from scone_b200 import _lib
    L = _lib.load()
    rng = np.random.default_rng(0)
    table = rng.integers(0, 256, size=(1000, 96), dtype=np.uint8)
    ids = rng.integers(0, 1000, size=777).astype(np.int32)
    for threads in (1, 3, 16):
        out = np.zeros((777, 96), dtype=np.uint8)
        rc = L.scone_host_gather_rows(table.ctypes.data, 96, 1000, ids.ctypes.data, 777, out.ctypes.data, threads)
        assert rc == 0 and np.array_equal(out, table[ids])
    bad = ids.copy()
    bad[5] = 1000
    assert L.scone_host_gather_rows(table.ctypes.data, 96, 1000, bad.ctypes.data, 777, out.ctypes.data, 4) == _lib.E_INVALID
    assert b"outside" in L.scone_last_error()
    assert L.scone_host_gather_rows(table.ctypes.data, 96, 1000, ids.ctypes.data, 0, out.ctypes.data, 4) == 0


def test_c_abi_rejects_bad_arguments_without_a_gpu():
    """Argument validation happens before any CUDA call, so it can be exercised here."""
    import ctypes as C
    from scone_b200 import _lib
    L = _lib.load()
    rs, so = C.c_int64(), C.c_int32()
    assert L.scone_table_layout(1, 1024, 128, 0, C.byref(rs), C.byref(so)) == 0 and (rs.value, so.value) == (1056, 1024)
    assert L.scone_table_layout(2, 4096, 128, 128, C.byref(rs), C.byref(so)) == 0 and (rs.value, so.value) == (2176, 2048)
    assert L.scone_table_layout(3, 1024, 128, 0, C.byref(rs), C.byref(so)) == 0 and (rs.value, so.value) == (4096, 0)   # SCONE_QUANT_FP32
    assert L.scone_table_layout(7, 1024, 128, 0, C.byref(rs), C.byref(so)) == _lib.E_INVALID
    assert L.scone_table_layout(2, 1000, 128, 0, C.byref(rs), C.byref(so)) == _lib.E_INVALID
    h = C.c_void_p()
    assert L.scone_index_create(None, None, 5, 9, 0.5, None, C.byref(h)) == _lib.E_INVALID        # max_n > 7
    assert b"max_n" in L.scone_last_error()
    assert L.scone_index_create(None, None, 5, 3, 0.95, None, C.byref(h)) == _lib.E_INVALID       # load factor
    assert L.scone_index_lookup(None, None, 1, 1, None, None, None) == _lib.E_INVALID
    assert L.scone_index_destroy(None) == 0 and L.scone_pipeline_destroy(None) == 0
    assert L.scone_pipeline_follow(None, None) == _lib.E_INVALID
    opts = _lib.EmbedOpts(0x80)                                                                   # unknown flag bit
    assert L.scone_embed_forward_ex(None, None, None, 0, None, None, 1, 1, None, 0, None, None, None, C.byref(opts), None) == _lib.E_INVALID
    assert b"flag" in L.scone_last_error()
    desc = _lib.TableDesc(16, 100, 4, 1, 1024, 128, 1024)                                         # row_stride 100: not a multiple of 16
    assert L.scone_table_gather(C.byref(desc), None, 1, None, 2, None, None) == _lib.E_INVALID
    # the projection fold's TMA row coordinates are 32-bit: k = 2^31 source rows is refused (aligned stand-in pointers, never read)
    desc = _lib.TableDesc(256, 1056, 4, 1, 1024, 128, 1024)
    assert L.scone_table_store_projected(C.byref(desc), 512, 768, 64, 1024, 0, 1 << 31, None, None) == _lib.E_INVALID
    assert b"k too large" in L.scone_last_error()


def test_every_table_layout_is_accepted_by_the_table_check():
    """scone_table_layout and the descriptor check of every table entry point state one row-format rule: each layout is
    accepted, a row_stride 16 bytes short of the row is refused, and INT8 / INT4 scales may sit at any aligned offset past
    the payload.  check_table runs before scone_table_gather's k == 0 return, so no call reaches the device."""
    import ctypes as C
    from scone_b200 import _lib
    L = _lib.load()
    rows = 16                                                    # aligned stand-in pointer, never read

    def layout(quant, dim, group, align):
        rs, so = C.c_int64(), C.c_int32()
        assert L.scone_table_layout(quant, dim, group, align, C.byref(rs), C.byref(so)) == 0, L.scone_last_error()
        return rs.value, so.value

    def check(quant, dim, group, stride, soff):
        desc = _lib.TableDesc(rows, stride, 1000, quant, dim, group, soff)
        return L.scone_table_gather(C.byref(desc), None, 0, None, _lib.OUT_FP32, None, None)

    cases = 0
    for name, quant in _lib.QUANT.items():
        for dim in (8, 64, 136, 1024, 4096, 16384):
            groups = [g for g in (8, 16, 32, 64, 128, 256) if dim % g == 0] if name == "int4" else [128]
            for group in groups:
                tight, soff = layout(quant, dim, group, 16)      # the smallest 16-byte multiple that holds the row
                for align in (16, 32, 128):
                    stride, soff_a = layout(quant, dim, group, align)
                    assert soff_a == soff and stride % align == 0 and tight <= stride < tight + align
                    assert check(quant, dim, group, stride, soff) == 0, (name, dim, group, align, L.scone_last_error())
                    cases += 1
                assert check(quant, dim, group, tight - 16, soff) == _lib.E_INVALID, (name, dim, group)
                assert b"row_stride" in L.scone_last_error()
                if name in ("int8", "int4"):
                    salign = 4 if name == "int8" else 2
                    roomy = tight + 128                          # room for the scales wherever they move
                    assert check(quant, dim, group, roomy, soff + salign) == 0, (name, dim, group)
                    for bad in (soff - salign, soff + 1):       # below the payload / misaligned
                        assert check(quant, dim, group, roomy, bad) == _lib.E_INVALID, (name, dim, group, bad)
                        assert b"scale_offset" in L.scone_last_error()
    assert cases == 3 * (3 * 6 + 24)


def test_bench_reference_arm_runs_on_cpu():
    """`bench.py --impl reference` (the CPU arm) needs no GPU and prints the contract's JSON line."""
    import json
    import subprocess
    import sys
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "config1", "--steps", "2",
                          "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "tokens/s" and line["value"] > 0 and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["steps"] == 2
    # other ranks of a torchrun launch exit quietly
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "config1",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
    # the dump belongs to the GPU arm, and a run needs at least one timed step
    for extra in (["--impl", "reference", "--dump-outputs", "x"], ["--workload", "config5", "--dump-outputs", "x"], ["--steps", "0"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120)
        assert out.returncode == 2 and "error" in out.stderr


@pytest.mark.gpu
def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """`bench.py --dump-outputs DIR` writes the results of the last timed step as float32 / float64 within 64 MB.  The steps
    rotate over 8 seeded id batches (step k runs batch k % 8), so 2 and 10 steps both end on batch 1 and 1 step on batch 0:
    the first two dumps are identical, the third differs, and batch 1's dump is checked against the oracle on inputs rebuilt
    here from bench.py's seeds (vocabulary seed 0, table seed 2, fallback rows seed 3, batch k seed 100 + k)."""
    import subprocess
    import sys
    from oracle.c_oracle import COracleIndex
    from scone_b200.utils import synthetic as S
    dumps = {}
    for steps in ("2", "10", "1"):
        d = tmp_path / steps
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "config1", "--steps", steps, "--warmup", "1",
                              "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        assert sorted(os.listdir(d)) == ["embeddings.npy", "fgram_id.npy", "match_len.npy"]
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= 64 << 20
        dumps[steps] = {f[:-4]: np.load(d / f) for f in os.listdir(d)}
    z = dumps["2"]
    assert z["fgram_id"].dtype == np.float64 and z["match_len"].dtype == np.float32 and z["embeddings"].dtype == np.float32
    assert z["fgram_id"].shape == z["match_len"].shape == (8, 512) and z["embeddings"].shape == (8 * 512, 768)
    for k in z:
        assert np.array_equal(z[k], dumps["10"][k]), k
    assert not np.array_equal(z["fgram_id"], dumps["1"]["fgram_id"])
    # config1: N = 100 000 f-grams, max_n = 3, V = 50 257, D = 768, FP16 table, batch 8 x 512, bf16 output
    N, max_n, V, D, B, L = 100_000, 3, 50_257, 768, 8, 512
    toks, lens, longest = S.make_vocab_device(N, max_n, V, seed=0, device="cuda", return_longest=True)
    q = S.make_stream_device(toks, lens, B, L, V, seed=101, p_plant=1.0, pick_ids=longest).cpu().numpy()
    wid, wlen = COracleIndex(toks.cpu().numpy(), lens.cpu().numpy()).match(q, nthreads=4)
    assert (wid >= 0).any() and (wid < 0).any()
    assert np.array_equal(z["fgram_id"], wid) and np.array_equal(z["match_len"], wlen)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(2)
    rows = torch.randn((N, D), generator=gen, device="cuda", dtype=torch.float32) * 0.02
    hit = wid >= 0
    want = np.empty((B, L, D), np.uint16)
    want[hit] = po.cast_bits(po.OracleTable.from_fp32(rows[torch.from_numpy(wid[hit].astype(np.int64)).cuda()].cpu().numpy(), "fp16")
                             .rows_fp32(np.arange(int(hit.sum()))), "bf16")
    base = S.make_base_device(V, D, torch.bfloat16, seed=3, device="cuda").view(torch.int16).cpu().numpy().view(np.uint16)
    want[~hit] = base[q[~hit]]
    assert np.array_equal(z["embeddings"], po.bf16_bits_to_f32(want).reshape(B * L, D))


def test_extractor_map_assignment_like_reference_load():
    """The reference lets callers assign the three maps (its own load() does, n_gram_extractor.py:159-165)."""
    from scone_b200 import NGramExtractor
    ex = NGramExtractor(max_n=3, min_freq=1, max_f_grams=10)
    ex.f_gram_to_id = {(5, 6): 1, (7,): 0, (1, 2, 3): 2}
    assert ex.id_to_f_gram == {0: (7,), 1: (5, 6), 2: (1, 2, 3)} and ex.f_grams == {(7,), (5, 6), (1, 2, 3)}
    t, l = ex.vocab_arrays()
    assert t.tolist() == [[7, -1, -1], [5, 6, -1], [1, 2, 3]] and l.tolist() == [1, 2, 3] and len(ex) == 3
    ex.id_to_f_gram = {0: (9, 9)}
    assert ex.f_gram_to_id == {(9, 9): 0}
    with pytest.raises(ValueError):
        ex.f_gram_to_id = {(1,): 0, (2,): 5}          # ids must be dense
    ex.f_gram_to_id = {(1, 2, 3, 4): 0}                # longer than max_n: can never match in the reference either
    import torch
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="longer than max_n"):
            ex.device_index()


def test_reads_extractor_file_written_by_the_reference():
    """tests/golden/ref_extractor.npy was written by the unmodified reference's NGramExtractor.save."""
    from scone_b200 import NGramExtractor
    z = load_golden("cache_small.npz")
    ex = NGramExtractor.load(os.path.join(ROOT, "tests", "golden", "ref_extractor.npy"))
    t, l = ex.vocab_arrays()
    assert ex.max_n == int(z["max_n"]) and np.array_equal(l, z["vocab_lens"])
    assert np.array_equal(t[:, :z["vocab_tokens"].shape[1]], z["vocab_tokens"])


def test_bench_byte_accounting_matches_the_survey_formula():
    """SURVEY.md 8d: bytes/token = 8 + slot_bytes * P + h R + (1 - h) 2D + 2D + 5, R = 2D | D + 4 | D/2 + 2 D/128."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    assert b.row_bytes_algorithmic("fp16", 768) == 1536 and b.row_bytes_algorithmic("fp32", 768) == 3072
    assert b.row_bytes_algorithmic("int8", 1024) == 1028
    assert b.row_bytes_algorithmic("int4", 4096) == 2112
    w2, w3 = b.WORKLOADS["config2"], b.WORKLOADS["config3"]
    # with the survey's 16-byte slots and h = 1 these are exactly its table entries (3 153 and 10 397 B/token)
    assert b.bytes_per_token(w2, 1.0, 4, slot_bytes=16) == 8 + 64 + 1028 + 2048 + 5 == 3153
    assert b.bytes_per_token(w3, 1.0, 5, slot_bytes=16) == 8 + 80 + 2112 + 8192 + 5 == 10397
    assert b.bytes_per_token(w2, 0.75, 3) == 8 + 96 + 0.75 * 1028 + 0.25 * 2048 + 2048 + 5


def test_compact20_slot_packing_is_injective():
    """numpy restatement of index_format.cuh::Compact20Slot::pack (a 28-bit id + five 20-bit tokens, reverse order, 0xFFFFF padded, in 16 bytes):
    the four words determine (length, tokens) uniquely and the id survives next to the four spare token bits; the all-ones word
    that marks an empty slot cannot be produced by a valid entry (ids < 2^28 - 1)."""
    PAD = 0xFFFFF
    rng = np.random.default_rng(20)

    def pack(fid, toks_rev):
        t = [int(x) for x in toks_rev] + [PAD] * (5 - len(toks_rev))
        w0 = (fid & 0x0FFFFFFF) | ((t[0] & 0xF) << 28)
        w1 = (t[0] >> 4) | ((t[1] & 0xFFFF) << 16)
        w2 = (t[1] >> 16) | (t[2] << 4) | ((t[3] & 0xFF) << 24)
        w3 = (t[3] >> 8) | (t[4] << 12)
        assert max(w0, w1, w2, w3) < 2 ** 32
        return w0, w1, w2, w3

    def unpack(w):
        w0, w1, w2, w3 = w
        t0 = (w0 >> 28) | ((w1 & 0xFFFF) << 4)
        t1 = (w1 >> 16) | ((w2 & 0xF) << 16)
        t2 = (w2 >> 4) & PAD
        t3 = (w2 >> 24) | ((w3 & 0xFFF) << 8)
        t4 = w3 >> 12
        toks = [t for t in (t0, t1, t2, t3, t4)]
        while toks and toks[-1] == PAD:
            toks.pop()
        return w0 & 0x0FFFFFFF, toks

    seen = {}
    for _ in range(20000):
        n = int(rng.integers(1, 6))
        toks = rng.integers(0, PAD, size=n).tolist()              # valid tokens are < 0xFFFFF
        fid = int(rng.integers(0, 2 ** 28 - 1))
        w = pack(fid, toks)
        assert w[0] != 0xFFFFFFFF
        assert unpack(w) == (fid, toks)
        key = (w[0] >> 28, w[1], w[2], w[3])
        assert seen.setdefault(key, toks) == toks                 # equal key words <=> equal (length, tokens)
    assert pack(2 ** 28 - 2, [PAD - 1] * 5)[0] != 0xFFFFFFFF


def test_fold_reciprocal_division_is_the_correctly_rounded_quotient():
    """csrc/fold.cu divides by a per-row scale as: refined reciprocal once (rcp seed, one Newton step), then per element
    q = a*y; r = fma(-b, q, a); q = fma(r, y, q); r = fma(-b, q, a); q = fma(r, y, q) -- and claims the result IS the IEEE quotient
    (the oracle's `x / s`).  Checked here in exact rational arithmetic (every fma rounded once, to nearest even, 24-bit
    significand), for reciprocal seeds up to 2 ulp off (the hardware's rcp.approx is within 1), on random operands and on the
    adversarial ones: quotients at and next to the .5 ties that `rint` would flip."""
    from fractions import Fraction as F
    import random

    def rn32(x):                                    # exact rational -> nearest binary32 (as a Fraction); normal range only
        if x == 0:
            return F(0)
        s, a = (1, x) if x > 0 else (-1, -x)
        e = a.numerator.bit_length() - a.denominator.bit_length()
        if F(2) ** e > a:
            e -= 1
        assert F(2) ** e <= a < F(2) ** (e + 1) and -100 < e < 100
        ulp = F(2) ** (e - 23)
        n, rem = divmod(a, ulp)
        if rem * 2 > ulp or (rem * 2 == ulp and n % 2 == 1):
            n += 1
        return s * n * ulp

    def ulp_of(x):
        e = x.numerator.bit_length() - x.denominator.bit_length()
        if F(2) ** e > abs(x):
            e -= 1
        return F(2) ** (e - 23)

    def fold_div(a, b, seed_off):
        y0 = rn32(1 / b)
        y0 += seed_off * ulp_of(y0)
        e = rn32(1 - b * y0)
        y = rn32(y0 + y0 * e)
        q = rn32(a * y)
        r = rn32(a - b * q)
        q = rn32(q + r * y)
        r = rn32(a - b * q)
        return rn32(q + r * y)

    rng = random.Random(7)
    cases = []
    for _ in range(800):
        amax = rn32(F(rng.getrandbits(24) | (1 << 23)) * F(2) ** rng.randint(-60, 20))
        b = rn32(amax / 127)                        # the INT8 row scale; the INT4 group scale amax / 7 below
        if rng.random() < 0.3:
            b = rn32(amax / 7)
        for _ in range(6):
            cases.append((rn32(amax * F(rng.randint(-(1 << 24), 1 << 24), 1 << 24)), b))      # anywhere in [-amax, amax]
            k = rng.randint(-127, 126)
            tie = rn32((F(k) + F(1, 2)) * b)                                                    # a / b next to k + 0.5
            cases.append((tie, b))
            cases.append((tie + rng.choice((-1, 1)) * ulp_of(tie), b))
    bad = 0
    for a, b in cases:
        want = rn32(a / b)
        for off in (-2, -1, 0, 1, 2):
            bad += fold_div(a, b, off) != want
    assert bad == 0, f"{bad} of {5 * len(cases)} quotients are not correctly rounded"
