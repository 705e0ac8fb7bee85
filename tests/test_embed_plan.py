"""The fused path's launch plan (scone_b200/csrc/embed_plan.h), compiled on the host with g++.

The plan alone decides which kernel, shape, lanes per position and ring layout a call runs; these tests pin that choice for
the named workloads and check, over a grid of row geometries, the conditions the kernels rely on.
"""

import itertools

import pytest

from plan_driver import PlanDriver

SMS = 148


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    """plan(cases) -> one line per case; a case is (D, row_stride, pos, additive, resolved, P, SCONE_EMBED_PIPE or None, T)."""
    try:
        driver = PlanDriver.build(str(tmp_path_factory.mktemp("embed_plan")))
    except FileNotFoundError:
        pytest.skip("no host C++ compiler")
    return lambda cases: driver.plan(cases, SMS)


# (D, row_stride, position rows, additive, resolved ids, P, SCONE_EMBED_PIPE, T) -> the launch, recorded from the dispatch
# this plan replaced (row strides as table_layout gives them at align 32; P as lanes_per_position gives it for the vocabulary)
NAMED = {
    # bench.py configs, plain path
    "config1": ((768, 1536, 0, 0, 0, 2, None, 8 * 512),
                "bulk nm 4 nl 0 ng 4 minb 3 budget 71680 P 4 add 0 ring 5 slot 1536 smem 62720 stagger 0 grid 444 threads 256"),
    "config2": ((1024, 1056, 0, 0, 0, 4, None, 64 * 1024),
                "bulk nm 4 nl 0 ng 4 minb 3 budget 71680 P 4 add 0 ring 4 slot 2048 smem 66816 stagger 500 grid 444 threads 256"),
    "config3": ((4096, 2112, 0, 0, 0, 4, None, 256 * 2048),
                "bulk nm 6 nl 0 ng 12 minb 1 budget 204800 P 8 add 0 ring 6 slot 8192 smem 197376 stagger 0 grid 148 threads 576"),
    "config5": ((2048, 2080, 0, 0, 0, 4, None, 256 * 2048),
                "bulk nm 6 nl 0 ng 12 minb 1 budget 204800 P 4 add 0 ring 6 slot 4096 smem 197888 stagger 0 grid 148 threads 576"),
    # extra rows per position: the pipeline
    "config2 + wpe": ((1024, 1056, 1, 0, 0, 4, None, 64 * 1024),
                      "pipe nm 6 nl 1 ng 4 minb 3 budget 71680 P 4 add 0 ring 2 meta 24 slot 2048 add_off 0 pos_off 16384 tile 32768 "
                      "smem 69760 stagger 500 grid 444 threads 352"),
    "config2 + base": ((1024, 1056, 0, 1, 0, 4, None, 64 * 1024),
                       "pipe nm 6 nl 1 ng 4 minb 3 budget 71680 P 4 add 1 ring 2 meta 24 slot 4096 add_off 2048 pos_off 0 tile 32768 "
                       "smem 69760 stagger 500 grid 444 threads 352"),
    "config2 + both": ((1024, 1056, 1, 1, 0, 4, None, 64 * 1024),
                       "pipe nm 4 nl 2 ng 8 minb 2 budget 112640 P 4 add 1 ring 2 meta 16 slot 4096 add_off 2048 pos_off 32768 tile 49152 "
                       "smem 102528 stagger 0 grid 296 threads 448"),
    "config3 + wpe": ((4096, 2112, 1, 0, 0, 4, None, 256 * 2048),
                      "pipe nm 6 nl 4 ng 12 minb 1 budget 204800 P 8 add 0 ring 3 meta 24 slot 8192 add_off 0 pos_off 32768 tile 65536 "
                      "smem 199168 stagger 0 grid 148 threads 704"),
    "config3 + base": ((4096, 2112, 0, 1, 0, 4, None, 256 * 2048),
                       "pipe nm 6 nl 4 ng 12 minb 1 budget 204800 P 8 add 1 ring 3 meta 24 slot 16384 add_off 8192 pos_off 0 tile 65536 "
                       "smem 199168 stagger 0 grid 148 threads 704"),
    "config3 + both": ((4096, 2112, 1, 1, 0, 4, None, 256 * 2048),
                       "pipe nm 6 nl 4 ng 12 minb 1 budget 204800 P 8 add 1 ring 2 meta 24 slot 16384 add_off 8192 pos_off 65536 tile 98304 "
                       "smem 199168 stagger 0 grid 148 threads 704"),
    # fp32 rows (the reference's own format): 3-6 KB rows take the pipeline on the plain path too
    "fp32 D 768": ((768, 3072, 0, 0, 0, 4, None, 64 * 1024),
                   "pipe nm 5 nl 2 ng 4 minb 3 budget 71680 P 4 add 0 ring 2 meta 20 slot 3072 add_off 0 pos_off 0 tile 24576 "
                   "smem 53376 stagger 500 grid 444 threads 352"),
    "fp32 D 1024": ((1024, 4096, 0, 0, 0, 4, None, 64 * 1024),
                    "pipe nm 5 nl 2 ng 4 minb 3 budget 71680 P 4 add 0 ring 2 meta 20 slot 4096 add_off 0 pos_off 0 tile 32768 "
                    "smem 69760 stagger 500 grid 444 threads 352"),
    "fp32 D 1536": ((1536, 6144, 0, 0, 0, 4, None, 64 * 1024),
                    "pipe nm 4 nl 2 ng 8 minb 2 budget 112640 P 4 add 0 ring 2 meta 16 slot 6144 add_off 0 pos_off 0 tile 49152 "
                    "smem 102528 stagger 0 grid 296 threads 448"),
    # the shapes of test_embed_forward_rows_too_wide_for_the_ring (B 2 x L 75)
    "fp16 D 8192": ((8192, 16384, 0, 0, 0, 4, None, 150),
                    "bulk nm 3 nl 0 ng 12 minb 1 budget 204800 P 8 add 0 ring 3 slot 16384 smem 197376 stagger 0 grid 38 threads 480"),
    "int8 D 16384": ((16384, 16416, 0, 0, 0, 2, None, 150),
                     "ldg nm 2 nl 0 ng 6 minb 4 budget 0 P 2 add 0 smem 0 stagger 0 grid 10 threads 256"),
    "int4 D 16384": ((16384, 8448, 0, 0, 0, 2, None, 150),
                     "ldg nm 2 nl 0 ng 6 minb 4 budget 0 P 2 add 0 smem 0 stagger 0 grid 10 threads 256"),
    "fp16 D 4096": ((4096, 8192, 0, 0, 0, 1, None, 150),
                    "bulk nm 6 nl 0 ng 12 minb 1 budget 204800 P 8 add 0 ring 6 slot 8192 smem 197376 stagger 0 grid 38 threads 576"),
    # scone_embed_gather: ids already resolved, P = 4 whatever P says
    "gather config2": ((1024, 1056, 0, 0, 1, 1, None, 64 * 1024),
                       "bulk nm 4 nl 0 ng 4 minb 3 budget 71680 P 4 add 0 ring 4 slot 2048 smem 66816 stagger 500 grid 444 threads 256"),
    "gather config2 + wpe": ((1024, 1056, 1, 0, 1, 8, None, 64 * 1024),
                             "pipe nm 6 nl 1 ng 4 minb 3 budget 71680 P 4 add 0 ring 2 meta 24 slot 2048 add_off 0 pos_off 16384 tile 32768 "
                             "smem 69760 stagger 500 grid 444 threads 352"),
    # SCONE_EMBED_PIPE forces the kernel of the plain path ...
    "config2, SCONE_EMBED_PIPE=1": ((1024, 1056, 0, 0, 0, 4, "1", 64 * 1024),
                                    "pipe nm 5 nl 2 ng 4 minb 3 budget 71680 P 4 add 0 ring 4 meta 20 slot 2048 add_off 0 pos_off 0 tile 16384 "
                                    "smem 69760 stagger 500 grid 444 threads 352"),
    "config3, SCONE_EMBED_PIPE=1": ((4096, 2112, 0, 0, 0, 4, "1", 256 * 2048),
                                    "pipe nm 6 nl 4 ng 12 minb 1 budget 204800 P 4 add 0 ring 3 meta 24 slot 8192 add_off 0 pos_off 0 tile 65536 "
                                    "smem 200832 stagger 0 grid 148 threads 704"),
    "fp32 D 1024, SCONE_EMBED_PIPE=0": ((1024, 4096, 0, 0, 0, 4, "0", 64 * 1024),
                                        "bulk nm 6 nl 0 ng 12 minb 1 budget 204800 P 4 add 0 ring 6 slot 4096 smem 197888 stagger 0 grid 148 "
                                        "threads 576"),
    # ... and leaves extra rows on the pipeline
    "config2 + both, SCONE_EMBED_PIPE=0": ((1024, 1056, 1, 1, 0, 4, "0", 64 * 1024),
                                           "pipe nm 4 nl 2 ng 8 minb 2 budget 112640 P 4 add 1 ring 2 meta 16 slot 4096 add_off 2048 "
                                           "pos_off 32768 tile 49152 smem 102528 stagger 0 grid 296 threads 448"),
}


def test_plan_of_the_named_workloads(plan):
    got = plan([case for case, _ in NAMED.values()])
    for (name, (_, want)), line in zip(NAMED.items(), got):
        assert line == want, name


def _fields(line):
    w = line.split()
    return w[0], {k: int(v) for k, v in zip(w[1::2], w[2::2])}


def test_plan_invariants_over_a_grid_of_row_geometries(plan):
    cases = []
    for D in list(range(8, 16385, 248)) + [768, 1024, 2048, 4096, 8192, 16384]:
        strides = {(b + a - 1) // a * a for b in (D // 2 + 2 * (D // 8), D + 4, 2 * D, 4 * D) for a in (32, 128)}
        strides |= set(range((D // 2 + 15) // 16 * 16, 4 * D + 65537, 1552))
        for rs, pos, add, P, env in itertools.product(sorted(strides), (0, 1), (0, 1), (1, 2, 4, 8), (None, "0", "1")):
            cases.append((D, rs, pos, add, 0, P, env, 300000))
    lines = plan(cases)
    seen = set()
    for (D, rs, pos, add, res, P, env, T), line in zip(cases, lines):
        fam, f = _fields(line)
        seen.add((fam, f["nm"], f["ng"], f["minb"], f["P"], f["add"]))
        G = 32 // f["P"]
        assert f["P"] >= P and (not add or f["P"] >= 4), line
        assert f["add"] == add, line
        assert f["threads"] == 32 * (f["nm"] + f["nl"] + f["ng"]), line
        assert f["grid"] == min((T + G - 1) // G, SMS * f["minb"]), line
        assert f["smem"] <= f["budget"], line
        if fam == "bulk":
            assert not pos and not add, "the single-ring kernel serves the plain path only: " + line
            assert f["ring"] >= 2 and f["ring"] >= f["nm"] and f["ring"] <= 16, line
            assert f["slot"] >= max(rs, 2 * D) and f["slot"] % 128 == 0, line
        elif fam == "pipe":
            assert 2 <= f["ring"] <= 16, line
            assert f["tile"] <= (1 << 20) - 16, line
            assert f["meta"] % f["nm"] == 0 and f["meta"] <= 32, line
            assert f["nl"] <= G, line
            assert f["slot"] >= max(rs, 2 * D) + (2 * D if add else 0), line
            assert (f["pos_off"] > 0) == bool(pos) and (f["add_off"] > 0) == bool(add), line
        else:
            assert fam == "ldg" and f["smem"] == 0, line
    assert {fam for fam, *_ in seen} == {"bulk", "pipe", "ldg"}
