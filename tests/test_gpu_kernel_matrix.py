"""Every fused-path kernel the library compiles, run past its ring wrap-around and checked bit for bit.

embed_inst.cu compiles exactly the (shape row, P, ADD) combinations that kShapes in embed_plan.h lists, per (table format,
output type).  The kernels synchronise through parity-only mbarriers, and what keeps a waiter from passing a barrier one
phase too early (ring >= NM, a single-ring slot refilled by different matchers when ring % NM != 0, a metadata ring that is
a multiple of NM, every gather warp releasing every tile) only matters once a CTA has gone round its ring.  So for every
compiled instance this file finds a real call the plan sends there (on the CPU, through tests/plan_driver.py), sizes it so
that every CTA goes round its rings at least twice, with a ragged last CTA and a ragged last tile, and checks the whole
output against a plain torch restatement and the C oracle.  A small case (one tile per CTA, partial grid) runs as well.
"""

from __future__ import annotations

import functools
import os

import numpy as np
import pytest

from plan_driver import PlanDriver

QUANTS = ("fp32", "fp16", "int8", "int4")
OUTS = ("bf16", "fp16")
QUANT_ID = {"fp16": 0, "int8": 1, "int4": 2, "fp32": 3}       # SCONE_QUANT_* (the kernels' QUANT template argument)
OUT_ID = {"bf16": 0, "fp16": 1}                               # SCONE_OUT_*
LDG_RING = 16                 # embed_kernel's ring (kRing in embed_kernels.cuh)
MAX_D = 16384
CPU_SMS = 148                 # sizes checked on the CPU are for a B200; the GPU items use the device's own SM count
ENVS = (None, "0", "1")       # SCONE_EMBED_PIPE
INDEX_FORMATS = (None, "wide", "prefer-compact20")   # SCONE_INDEX_FORMAT, cycled across cases

# lanes per position (lanes_per_position in match.cuh) -> the f-gram lengths of a vocabulary that needs exactly that many
LENGTHS = {1: (1,), 2: (1, 2), 4: (1, 2, 3), 8: (1, 2, 3, 4, 5)}

# Compiled for every format, but no call of that format is ever planned onto them: searched over every D <= 16 384 (every
# multiple of 128 for INT4) at table align 32 and 128, every P, with and without position rows and the additive combine, and
# SCONE_EMBED_PIPE unset / 0 / 1.  Pruning them is a library change; listing them here makes a change of kShapes or of the
# plan that adds or removes one fail loudly.
UNREACHABLE = {
    ("fp32", (5, 8, 0)): "kBulkMid at P 8: cannot be planned for FP32 rows",
    ("fp16", (5, 8, 0)): "kBulkMid at P 8: cannot be planned for FP16 rows",
    ("int8", (5, 8, 0)): "kBulkMid at P 8: cannot be planned for INT8 rows",
    ("int4", (2, 4, 0)): "kBulkWide at P 4: cannot be planned for INT4 rows",
}


def row_stride(quant: str, D: int, align: int, group: int = 128) -> int:
    """scone_table_layout's row stride: the stored row (INT8 + fp32 scale, INT4 + one fp16 scale per group) rounded up."""
    need = {"fp32": 4 * D, "fp16": 2 * D, "int8": D + 4, "int4": D // 2 + 2 * (D // group)}[quant]
    return (need + align - 1) // align * align


@functools.lru_cache(maxsize=None)
def driver() -> PlanDriver:
    return PlanDriver.build()


@functools.lru_cache(maxsize=None)
def shapes():
    return {s.row: s for s in driver().shapes()}


def compiled_instances():
    return sorted(i for s in shapes().values() for i in s.instances())


class Case:
    """A call that the plan sends to one instance: table geometry, vocabulary P, position rows, additive, SCONE_EMBED_PIPE."""

    def __init__(self, quant, D, align, P, pos, add, env):
        self.quant, self.D, self.align, self.P, self.pos, self.add, self.env = quant, D, align, P, pos, add, env
        self.stride = row_stride(quant, D, align)

    def call(self, T, resolved=False):
        return (self.D, self.stride, self.pos, self.add, int(resolved), self.P, self.env, T)

    def __repr__(self):
        return f"{self.quant} D {self.D} align {self.align} P {self.P} pos {self.pos} add {self.add} SCONE_EMBED_PIPE {self.env}"


@functools.lru_cache(maxsize=None)
def search():
    """{(quant, instance): [case, ...]}: the smallest-D call reaching each instance, for pipeline instances one with and
    one without position rows where both reach it."""
    found = {}
    for quant in QUANTS:
        cands = [Case(quant, D, align, P, pos, add, env)
                 for D in range(128 if quant == "int4" else 8, MAX_D + 1, 128 if quant == "int4" else 8)
                 for align in (32, 128) for P in (1, 2, 4, 8) for pos in (0, 1) for add in (0, 1) for env in ENVS]
        plans = driver().detail([c.call(1 << 20) for c in cands], CPU_SMS)
        for c, pl in zip(cands, plans):
            per = found.setdefault((quant, pl.instance), {})
            if c.pos not in per:          # candidates come in increasing D: the first one is the smallest
                per[c.pos] = c
    out = {}
    for (q, inst), per in found.items():
        cases = [per[p] for p in sorted(per)]
        out[(q, inst)] = cases if shapes()[inst[0]].family == "pipe" else [min(cases, key=lambda c: c.D)]
    return out


def matrix():
    """[(quant, out, instance)] for every compiled instance a call of that format can reach."""
    reach = search()
    return [(q, o, inst) for q in QUANTS for o in OUTS for inst in compiled_instances() if (q, inst) in reach]


def wrap_ring(inst, pl):
    """Ring slots a CTA must go round: the row ring, and for the pipeline also its metadata ring."""
    fam = shapes()[inst[0]].family
    return LDG_RING if fam == "ldg" else max(pl.ring, pl.meta)


def sizes(case, inst, sms):
    """(B, L) of the wrap case and of the small case of `case` on `sms` SMs.

    Wrap: every CTA gets at least 2 R + 1 tiles (R = the larger ring), so each of its barriers completes at least two full
    phases; the last CTA gets fewer tiles than the others and the last tile fewer positions than G; L is not a multiple of
    G, so tiles straddle sequence ends.  Small: fewer tiles than the resident grid (one tile per CTA, a partial grid) and
    L < G, so that one tile spans several sequences."""
    s = shapes()[inst[0]]
    G = 32 // inst[1]
    resident = sms * s.minb
    pl = driver().detail([case.call(1 << 24)], sms)[0]
    R = wrap_ring(inst, pl)
    L = 97
    B = -(-(2 * R + 1) * resident * G // L)
    while True:
        T = B * L
        nt = -(-T // G)
        if T % G and nt % resident and nt >= (2 * R + 1) * resident + 1:
            break
        B += 1
    Ls = G - 1
    Bs = max(1, resident * G // (3 * Ls))
    return (B, L), (Bs, Ls)


def plan_for(case, B, L, sms, resolved=False):
    return driver().detail([case.call(B * L, resolved)], sms)[0]


# ---- the matrix, checked on the CPU -----------------------------------------------------------------------------------


def test_every_compiled_kernel_has_a_case():
    missing = sorted((q, inst) for q in QUANTS for inst in compiled_instances() if (q, inst) not in search())
    assert missing == sorted(UNREACHABLE), missing
    for (q, inst), cases in search().items():
        assert inst in compiled_instances(), (q, inst)
        for c in cases:
            pl = plan_for(c, 1, 4096, CPU_SMS)
            assert pl.instance == inst, (c, inst)
    per_pair = {}
    for q, o, inst in matrix():
        per_pair[(q, o)] = per_pair.get((q, o), 0) + 1
    assert per_pair == {(q, o): len(compiled_instances()) - 1 for q in QUANTS for o in OUTS}


def test_every_case_meets_the_size_rules():
    for q, _, inst in matrix():
        s = shapes()[inst[0]]
        for c in search()[(q, inst)]:
            (B, L), (Bs, Ls) = sizes(c, inst, CPU_SMS)
            G = 32 // inst[1]
            pl = plan_for(c, B, L, CPU_SMS)
            assert pl.instance == inst and pl.grid == CPU_SMS * s.minb, c
            R = wrap_ring(inst, pl)
            assert pl.num_tiles // pl.grid >= 2 * R + 1 and pl.num_tiles % pl.grid, c     # every CTA wraps twice; ragged last CTA
            assert (B * L) % G and L % G, c                                              # ragged last tile, straddled sequences
            assert (pl.stagger > 0) == bool(s.stagger), c
            small = plan_for(c, Bs, Ls, CPU_SMS)
            assert small.instance == inst and small.num_tiles < CPU_SMS * s.minb and small.grid == small.num_tiles, c
            assert Ls < G, c


def coverage():
    """{condition: {family: number of matrix items that reach it past at least one full ring wrap}}."""
    table = {k: {} for k in ("ring % nm != 0 (single ring)", "metadata-ring wrap (pipeline)", "matcher stagger", "ragged last CTA")}

    def bump(k, fam):
        table[k].setdefault(fam, set()).add((q, o, inst))

    for q, o, inst in matrix():
        s = shapes()[inst[0]]
        for c in search()[(q, inst)]:
            (B, L), _ = sizes(c, inst, CPU_SMS)
            pl = plan_for(c, B, L, CPU_SMS)
            if pl.num_tiles // pl.grid <= wrap_ring(inst, pl):
                continue
            if s.family == "bulk" and pl.ring % s.nm:
                bump("ring % nm != 0 (single ring)", s.family)
            if s.family == "pipe" and pl.num_tiles // pl.grid > pl.meta:
                bump("metadata-ring wrap (pipeline)", s.family)
            if pl.stagger:
                bump("matcher stagger", s.family)
            if pl.num_tiles % pl.grid:
                bump("ragged last CTA", s.family)
    return {k: {f: len(items) for f, items in v.items()} for k, v in table.items()}


def test_wrap_cases_reach_every_synchronisation_condition():
    t = coverage()
    fams = {s.family for s in shapes().values()}
    assert set(t["ring % nm != 0 (single ring)"]) == {"bulk"}
    assert set(t["metadata-ring wrap (pipeline)"]) == {"pipe"}
    assert set(t["matcher stagger"]) == {s.family for s in shapes().values() if s.stagger}
    assert set(t["ragged last CTA"]) == fams



# ---- the matrix on the GPU ----------------------------------------------------------------------------------------------

DEV = "cuda"
V_TOKENS = 4000               # token range of the streams; the base table has BASE_SHORT rows fewer
BASE_SHORT = 3
N_FGRAMS = 400                # f-grams (= table rows; 400 % 3 != 0 for the sharded stand-in)
CHUNK_BYTES = 1 << 29         # fp32 bytes of reference restated at a time


def _mods():
    import torch
    import scone_b200 as sb
    from scone_b200.utils import synthetic as S
    return torch, sb, S


def _bits16(torch, t):
    return t.contiguous().view(torch.int16)


def _kernel_args(name):
    """Template arguments of the fused kernel named in a profiler trace, as ints (demangled or mangled names)."""
    import re
    if name.startswith("_Z"):
        return [int(x) for x in re.findall(r"L[ib](\d+)E", name)]
    m = re.search(r"embed_(?:bulk_|pipe_)?kernel<([^>]*)>", name)
    args = [re.sub(r"\((?:int|bool)\)", "", a).strip() for a in m.group(1).split(",")]
    return [{"true": 1, "false": 0}[a] if a in ("true", "false") else int(a) for a in args]


def _expected_kernel(quant, out, inst):
    s = shapes()[inst[0]]
    q, o, P = QUANT_ID[quant], OUT_ID[out], inst[1]
    if s.family == "bulk":
        return "embed_bulk_kernel", [q, o, P, s.nm, s.ng, s.minb]
    if s.family == "pipe":
        return "embed_pipe_kernel", [q, o, P, s.nm, s.nl, s.ng, s.minb, inst[2]]
    return "embed_kernel", [q, o, P, 4, s.nm, s.ng, s.minb]          # reads the combine at run time


def _launched_kernels(torch, fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    import re
    return [e.name for e in prof.events() if re.search(r"embed_(bulk_|pipe_)?kernel", e.name)]


def _assert_kernel(torch, fn, quant, out, inst):
    names = _launched_kernels(torch, fn)
    assert len(names) == 1, names
    kname, args = _expected_kernel(quant, out, inst)
    assert (kname + "<" in names[0] or kname + "I" in names[0]) and _kernel_args(names[0]) == args, (names[0], kname, args)


def _vocab(S, P, seed):
    lens_set = LENGTHS[P]
    toks, lens = S.make_vocab_numpy(N_FGRAMS, lens_set[-1], V_TOKENS, seed=seed, min_n=1)
    assert sorted(set(lens.tolist())) == list(lens_set)
    # a unigram on the last token, which has no base row: an additive hit there needs a base row that does not exist
    last = V_TOKENS - 1
    if not ((lens == 1) & (toks[:, 0] == last)).any():
        k = int(np.flatnonzero(lens == 1)[0])
        toks[k, 0] = last
    return toks, lens


def _stream(S, toks, lens, B, L, seed, wrap):
    """Ids with a hit rate of about 0.7; the wrap case also carries ids the base table lacks, negative ids and ids above
    int32; every case carries the last token, whose unigram is in the vocabulary but which has no base row."""
    q = S.make_stream_numpy(toks, lens, B, L, V_TOKENS, seed=seed, p_plant=0.3)
    rng = np.random.default_rng(seed)
    T = B * L
    odd = [V_TOKENS - 1, V_TOKENS - 2, V_TOKENS - BASE_SHORT, -1, -7, 2 ** 31, 2 ** 40 + 3] if wrap else [V_TOKENS - 1]
    at = rng.choice(T, size=min(T, max(len(odd), T // 400)), replace=False)
    q.reshape(-1)[at] = np.resize(np.array(odd, np.int64), at.size)
    return q


def _restate(torch, t, base, pos, ids, fid, additive, dtype):
    """The fused path restated in torch on the GPU, for a block of batch rows: fp32 row of the hit (plus the base row under
    the additive combine), else the base row, else zero; plus the position row; one rounding to the output type.
    fid >= t.num_rows (resolved ids only) is a zero row."""
    Vb = base.shape[0]
    valid = (ids >= 0) & (ids < Vb)
    hit = (fid >= 0) & (fid < t.num_rows)
    rows = t.gather(torch.where(hit, fid, 0).reshape(-1).long(), torch.float32).view(*fid.shape, -1)
    b = base.float()[torch.where(valid, ids, 0)]
    x = torch.where(hit[..., None], rows, torch.where((valid & (fid == -1))[..., None], b, torch.zeros_like(b)))
    if additive:
        x = torch.where((hit & valid)[..., None], b + rows, x)
    if pos is not None:
        x = x + pos[:ids.shape[-1]].float()[None]
    return x.to(dtype)


def _assert_equal_to_restatement(torch, out, t, base, pos, ids, fid, additive):
    B, L, D = out.shape
    step = max(1, CHUNK_BYTES // (4 * L * D))
    for b0 in range(0, B, step):
        b1 = min(B, b0 + step)
        want = _restate(torch, t, base, pos, ids[b0:b1], fid[b0:b1], additive, out.dtype)
        same = _bits16(torch, out[b0:b1]) == _bits16(torch, want)
        assert bool(same.all()), f"batch rows {b0}..{b1}: {int((~same).sum())} elements differ"


def _run(monkeypatch, quant, out, inst, case, B, L, index_format, wrap, seed):
    torch, sb, S = _mods()
    from oracle.c_oracle import COracleIndex
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    pl = plan_for(case, B, L, sms)
    assert pl.instance == inst, (case, B, L)
    for k, v in (("SCONE_EMBED_PIPE", case.env), ("SCONE_INDEX_FORMAT", index_format)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, v)
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[out]
    D = case.D
    toks, lens = _vocab(S, case.P, seed)
    q = _stream(S, toks, lens, B, L, seed + 1, wrap)
    rows = S.make_rows_numpy(N_FGRAMS, D, seed=seed + 2)
    base = S.make_base_device(V_TOKENS - BASE_SHORT, D, dtype, seed=seed + 3, device=DEV)
    pos = S.make_base_device(L + 3, D, dtype, seed=seed + 4, device=DEV) if case.pos else None
    ix = sb.FGramIndex(torch.from_numpy(toks).to(DEV), torch.from_numpy(lens).to(DEV))
    t = sb.CacheTable(N_FGRAMS, D, quant, align=case.align)
    assert t.row_stride == case.stride
    t.store(torch.from_numpy(rows).to(DEV))
    ids = torch.from_numpy(q).to(DEV)
    combine = "add" if case.add else "replace"
    status = torch.zeros(1, dtype=torch.int32, device=DEV)
    emb, fid, ml = sb.embed_forward(ix, t, base, ids, pos_emb=pos, status=status, combine=combine)
    torch.cuda.synchronize()
    # f-gram ids and match lengths of the whole batch
    wid, wlen = COracleIndex(toks, lens).match(q, nthreads=os.cpu_count() or 1)
    assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
    hit = float((wid >= 0).mean())
    assert 0.2 < hit < 0.9, hit
    # the whole output against the torch restatement
    _assert_equal_to_restatement(torch, emb, t, base, pos, ids, fid, case.add)
    # a base row that does not exist was needed exactly where the status bit says so
    valid = (q >= 0) & (q < V_TOKENS - BASE_SHORT)
    needs_base = (wid < 0) | ((wid >= 0) & bool(case.add))
    assert int(status.item()) == int((needs_base & ~valid).any())
    # a few batch rows against the C oracle: the first, the last, and the one where the last tile starts
    packed = t.storage.cpu().numpy()
    base_bits = _bits16(torch, base).cpu().numpy().view(np.uint16)
    pos_bits = _bits16(torch, pos).cpu().numpy().view(np.uint16) if pos is not None else None
    G = 32 // inst[1]
    for b in sorted({0, B - 1, (pl.num_tiles - 1) * G // L}):
        want, _, _, _ = COracleIndex(toks, lens).embed(quant, D, t.group, packed, t.row_stride, packed[:, t.scale_offset:] if t.scale_offset else None,
                                                       t.row_stride, base_bits, q[b:b + 1], out, pos_bits=pos_bits, additive=bool(case.add))
        assert np.array_equal(_bits16(torch, emb[b]).cpu().numpy().view(np.uint16), want[0]), b
    if wrap:
        # back to back with overlapped launches, into fresh zeroed buffers: the same bits
        outs = [(torch.zeros_like(emb), torch.zeros_like(fid), torch.zeros_like(ml)) for _ in range(2)]
        for o, i, m in outs:
            sb.embed_forward(ix, t, base, ids, pos_emb=pos, out=o, out_id=i, out_len=m, combine=combine, inputs_stable=True)
        torch.cuda.synchronize()
        for o, i, m in outs:
            assert torch.equal(_bits16(torch, o), _bits16(torch, emb)) and torch.equal(i, fid) and torch.equal(m, ml)
        del outs
    # the resolved-id path, where the plan sends it to the same kernel; f-gram ids past the table are zero rows + status
    if not case.add and plan_for(case, B, L, sms, resolved=True).instance == inst:
        rid = torch.from_numpy(wid).to(DEV)
        flat = rid.view(-1)
        bad = torch.arange(0, flat.numel(), max(1, flat.numel() // 5), device=DEV)
        flat[bad] = N_FGRAMS + bad.to(torch.int32) % 3
        st = torch.zeros(1, dtype=torch.int32, device=DEV)
        g = sb.embed_gather(t, base, ids, rid, pos_emb=pos, status=st)
        torch.cuda.synchronize()
        assert int(st.item()) == 1
        _assert_equal_to_restatement(torch, g, t, base, pos, ids, rid, False)
        del g
    # the launched kernel carries the template arguments the plan predicts
    _assert_kernel(torch, lambda: sb.embed_forward(ix, t, base, ids, pos_emb=pos, combine=combine), quant, out, inst)
    del emb


@pytest.mark.gpu
@pytest.mark.parametrize("quant,out,inst", [pytest.param(q, o, i, id=f"{q}-{o}-row{i[0]}-P{i[1]}-add{i[2]}") for q, o, i in matrix()])
def test_kernel_instance(monkeypatch, quant, out, inst):
    """One compiled kernel: each of its cases once past two ring wraps and once on a partial grid."""
    torch, _, _ = _mods()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    k = matrix().index((quant, out, inst))
    for n, case in enumerate(search()[(quant, inst)]):
        (B, L), (Bs, Ls) = sizes(case, inst, sms)
        _run(monkeypatch, quant, out, inst, case, B, L, INDEX_FORMATS[(k + n) % 3], True, seed=7 * k + n)
        torch.cuda.empty_cache()
        _run(monkeypatch, quant, out, inst, case, Bs, Ls, INDEX_FORMATS[(k + n + 1) % 3], False, seed=7 * k + n + 3)


class _SameDeviceShards:
    """The part of sharded.PeerShardedTable that embed_forward_sharded reads, with every shard on this device: row r of a
    table of `total_rows` rows is row r // W of shard r % W."""

    def __init__(self, sb, table, align, world):
        import torch
        self.world, self.total_rows, self.device = world, table.num_rows, table.device
        cap = -(-table.num_rows // world)
        self.shards = []
        for k in range(world):
            sh = sb.CacheTable(cap, table.dim, table.quant, table.group, align=align)
            assert sh.row_stride == table.row_stride
            mine = table.storage[k::world]
            sh.storage[:mine.shape[0]].copy_(mine)
            self.shards.append(sh)
        self.local = self.shards[0]
        self.ptr_table = torch.tensor([sh.storage.data_ptr() for sh in self.shards], dtype=torch.int64, device=self.device)


def _sharded_cases():
    """One case per family: single ring; pipeline with position rows; register-load."""
    picks = []
    for fam, want_pos in (("bulk", 0), ("pipe", 1), ("ldg", None)):
        cands = [(c.D, inst, c) for q, o, inst in matrix() if q == "int8" and o == "bf16" and shapes()[inst[0]].family == fam
                 and not inst[2] for c in search()[(q, inst)] if want_pos is None or c.pos == want_pos]
        _, inst, c = min(cands, key=lambda x: x[0])
        picks.append(pytest.param("int8", "bf16", inst, c, id=f"{fam}-int8-bf16-row{inst[0]}-P{inst[1]}"))
    return picks


@pytest.mark.gpu
@pytest.mark.parametrize("quant,out,inst,case", _sharded_cases())
def test_sharded_pointer_table_addressing(monkeypatch, quant, out, inst, case):
    """embed_forward_sharded reads row r from shard r % W at row r // W through the pointer table; with the shards on one
    device that is bit-identical to embed_forward on the unsharded table, for W = 1 and W = 3 (400 rows: a short last shard)."""
    torch, sb, S = _mods()
    from scone_b200 import sharded
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    (B, L), _ = sizes(case, inst, sms)
    if case.env is None:
        monkeypatch.delenv("SCONE_EMBED_PIPE", raising=False)
    else:
        monkeypatch.setenv("SCONE_EMBED_PIPE", case.env)
    dtype = {"bf16": torch.bfloat16, "fp16": torch.float16}[out]
    toks, lens = _vocab(S, case.P, 11)
    ids = torch.from_numpy(_stream(S, toks, lens, B, L, 12, True)).to(DEV)
    base = S.make_base_device(V_TOKENS - BASE_SHORT, case.D, dtype, seed=13, device=DEV)
    pos = S.make_base_device(L, case.D, dtype, seed=14, device=DEV) if case.pos else None
    ix = sb.FGramIndex(torch.from_numpy(toks).to(DEV), torch.from_numpy(lens).to(DEV))
    t = sb.CacheTable(N_FGRAMS, case.D, quant, align=case.align)
    t.store(torch.from_numpy(S.make_rows_numpy(N_FGRAMS, case.D, seed=15)).to(DEV))
    st = torch.zeros(1, dtype=torch.int32, device=DEV)
    want, wid, wlen = sb.embed_forward(ix, t, base, ids, pos_emb=pos, status=st)
    for world in (1, 3):
        shards = _SameDeviceShards(sb, t, case.align, world)
        st2 = torch.zeros(1, dtype=torch.int32, device=DEV)
        got, fid, ml = sharded.embed_forward_sharded(ix, shards, base, ids, pos_emb=pos, status=st2)
        torch.cuda.synchronize()
        assert torch.equal(fid, wid) and torch.equal(ml, wlen) and int(st2.item()) == int(st.item())
        assert torch.equal(_bits16(torch, got), _bits16(torch, want)), world
    _assert_kernel(torch, lambda: sharded.embed_forward_sharded(ix, shards, base, ids, pos_emb=pos), quant, out, inst)


# ---- INT4 group sizes other than 128 ----------------------------------------------------------------------------------

INT4_GROUPS = (8, 16, 32, 64, 256)
INT4_DIMS = (256, 4096, 16384)       # narrow rows; wide rows on the single ring and the pipeline; rows for the register-load kernel


def _int4_calls(D, group):
    """The calls of test_int4_group_sizes: (SCONE_EMBED_PIPE, position rows, additive) for a vocabulary with P = 4."""
    return [("0", 0, 0), ("1", 0, 0), (None, 1, 1)]


def test_int4_group_calls_reach_every_family():
    """The INT4 group items run every kernel family for every group size."""
    for group in INT4_GROUPS:
        fams = set()
        for D in INT4_DIMS:
            rs = row_stride("int4", D, 32, group)
            for env, pos, add in _int4_calls(D, group):
                pl = driver().detail([(D, rs, pos, add, 0, 4, env, 3 * 131)], CPU_SMS)[0]
                fams.add(shapes()[pl.row].family)
            assert shapes()[driver().detail([(D, rs, 0, 0, 1, 4, None, 3 * 131)], CPU_SMS)[0].row].family in fams
        assert fams == {"bulk", "pipe", "ldg"}, group


@pytest.mark.gpu
@pytest.mark.parametrize("D", INT4_DIMS)
@pytest.mark.parametrize("group", INT4_GROUPS)
def test_int4_group_sizes(monkeypatch, group, D):
    """INT4 tables with `group` elements per scale: the stored bytes are the oracle quantiser's, and the fused kernels, the
    position add with the additive combine, the resolved-id gather and the mean kernel equal the C / Python oracle."""
    torch, sb, S = _mods()
    from conftest import vocab_dict
    from oracle import py_oracle as po
    from oracle.c_oracle import COracleIndex
    if D % group:
        pytest.skip("D must be a multiple of the group")
    N, V, B, L, max_n = N_FGRAMS, V_TOKENS, 3, 131, 3
    toks, lens = _vocab(S, 4, group)
    q = S.make_stream_numpy(toks, lens, B, L, V, seed=group + 1, p_plant=0.3)
    rows = S.make_rows_numpy(N, D, seed=group + 2)
    rows[5, : group] *= 1e-7                # one group whose scale underflows fp16 (scale 1)
    tab = po.OracleTable.from_fp32(rows, "int4", group)
    packed, stride, soff = S.pack_table_numpy("int4", tab.payload, tab.scales)
    t = sb.CacheTable(N, D, "int4", group=group)
    assert (t.row_stride, t.scale_offset) == (stride, soff) and stride == row_stride("int4", D, 32, group)
    t.store(torch.from_numpy(rows).to(DEV))
    assert np.array_equal(t.storage.cpu().numpy(), packed)
    ix = sb.FGramIndex(torch.from_numpy(toks).to(DEV), torch.from_numpy(lens).to(DEV))
    cix = COracleIndex(toks, lens)
    base_bits = po.cast_bits(S.make_rows_numpy(V, D, seed=group + 3), "bf16")
    pos_bits = po.cast_bits(S.make_rows_numpy(L, D, seed=group + 4), "bf16")
    base = torch.from_numpy(base_bits.view(np.int16).copy()).view(torch.bfloat16).to(DEV)
    pos = torch.from_numpy(pos_bits.view(np.int16).copy()).view(torch.bfloat16).to(DEV)
    ids = torch.from_numpy(q).to(DEV)
    for env, with_pos, add in _int4_calls(D, group):
        if env is None:
            monkeypatch.delenv("SCONE_EMBED_PIPE", raising=False)
        else:
            monkeypatch.setenv("SCONE_EMBED_PIPE", env)
        want, wid, wlen, err = cix.embed("int4", D, group, packed, stride, packed[:, soff:], stride, base_bits, q, "bf16",
                                         pos_bits=pos_bits if with_pos else None, additive=bool(add))
        assert err == 0 and 0.2 < (wid >= 0).mean() < 0.9
        out, fid, ml = sb.embed_forward(ix, t, base, ids, pos_emb=pos if with_pos else None, combine="add" if add else "replace")
        torch.cuda.synchronize()
        assert np.array_equal(fid.cpu().numpy(), wid) and np.array_equal(ml.cpu().numpy(), wlen)
        assert np.array_equal(_bits16(torch, out).cpu().numpy().view(np.uint16), want), (env, with_pos, add)
    monkeypatch.delenv("SCONE_EMBED_PIPE", raising=False)
    want, wid, _, _ = cix.embed("int4", D, group, packed, stride, packed[:, soff:], stride, base_bits, q, "bf16")
    g = sb.embed_gather(t, base, ids, torch.from_numpy(wid).to(DEV))
    assert np.array_equal(_bits16(torch, g).cpu().numpy().view(np.uint16), want)
    m = sb.embed_mean_forward(ix, t, ids).cpu().numpy()
    g2i = vocab_dict(toks, lens)
    for b in range(B):
        np.testing.assert_allclose(m[b], po.assemble_mean(g2i, max_n, tab.rows_fp32, q[b].tolist(), D), rtol=0, atol=1e-8)


if __name__ == "__main__":
    # the coverage table, from the plan alone (B200: 148 SMs)
    print("| condition | " + " | ".join(f"{f} items" for f in ("bulk", "pipe", "ldg")) + " |")
    print("|---|---|---|---|")
    for k, v in coverage().items():
        print(f"| {k} | " + " | ".join(str(v.get(f, "-")) for f in ("bulk", "pipe", "ldg")) + " |")
