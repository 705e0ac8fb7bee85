"""The projection fold's launch plan (scone_b200/csrc/fold_plan.h), compiled on the host with g++.

The plan alone decides which fold path, cluster and grid a call of scone_table_store_projected runs; these tests pin that
choice for the named shapes and check, over a grid of calls, the conditions the kernels rely on.
"""

import itertools

import pytest

from plan_driver import PlanDriver

SMS = 148
FP16, INT8, INT4, FP32 = 0, 1, 2, 3


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    """plan(cases, sms) -> one line per case; a case is (quant, H, K, k, SCONE_FOLD_2SM, SCONE_FOLD_XCH, resident clusters)."""
    try:
        driver = PlanDriver.build(str(tmp_path_factory.mktemp("fold_plan")))
    except FileNotFoundError:
        pytest.skip("no host C++ compiler")
    return lambda cases, sms=SMS: driver.fold(cases, sms)


def _line(path, cluster, tiles, epi, stages, stage_bytes, box, n_chunks, k_blocks, m_groups, sweeps, grid, threads):
    return (f"{path} cluster {cluster} tiles {tiles} epi {epi} stages {stages} stage_bytes {stage_bytes} box {box} n_chunks {n_chunks} "
            f"k_blocks {k_blocks} m_groups {m_groups} sweeps {sweeps} grid {grid} threads {threads}")


SINGLE = ("single", 1, 1, 8, 4, 49152, 256)
PAIRS = ("pairs", 2, 2, 8, 4, 49152, 128)
PAIR_TILE = ("pairtile", 2, 2, 8, 6, 32768, 128)


def EXCHANGE(n):
    return ("exchange", n, 1, 16, 4, 49152, 256)


K_BENCH = 262144
# (quant, H, K = H_f, k, SCONE_FOLD_2SM, SCONE_FOLD_XCH, resident exchange clusters) -> the launch, recorded from the inline
# decision this plan replaced.  Residency as on a B200: 132 of the 148 SMs host clusters of up to 4 CTAs, 120 larger ones
# (DESIGN.md section 9: 33 clusters of 4, 15 of 8).
NAMED = {
    # tools/bench_fold.py
    "bench fp16 384 -> 768": ((FP16, 768, 384, K_BENCH, None, None, 33), _line(*PAIRS, 3, 6, 1024, 1, 148, 320)),
    "bench int8 384 -> 1024": ((INT8, 1024, 384, K_BENCH, None, None, 33), _line(*EXCHANGE(4), 4, 6, 2048, 1, 132, 576)),
    "bench int8 768 -> 1024": ((INT8, 1024, 768, K_BENCH, None, None, 33), _line(*EXCHANGE(4), 4, 12, 2048, 1, 132, 576)),
    "bench fp16 768 -> 1024": ((FP16, 1024, 768, K_BENCH, None, None, 33), _line(*PAIR_TILE, 4, 12, 1024, 1, 148, 320)),
    "bench int8 1024 -> 2048": ((INT8, 2048, 1024, K_BENCH, None, None, 15), _line(*EXCHANGE(8), 8, 16, 2048, 1, 120, 576)),
    "bench int4 1024 -> 4096": ((INT4, 4096, 1024, K_BENCH, None, None, 33), _line(*SINGLE, 16, 16, 2048, 1, 148, 320)),
    "bench fp16 1024 -> 4096": ((FP16, 4096, 1024, K_BENCH, None, None, 33), _line(*PAIR_TILE, 16, 16, 1024, 1, 148, 320)),
    "bench fp32 1024 -> 4096": ((FP32, 4096, 1024, K_BENCH, None, None, 33), _line(*SINGLE, 16, 16, 2048, 1, 148, 320)),
    # tests/test_gpu_parity.py::test_projection_fold shapes, INT8
    "test 384 -> 768, k 1000": ((INT8, 768, 384, 1000, None, None, 44), _line(*EXCHANGE(3), 3, 6, 8, 1, 24, 576)),
    "test 768 -> 1024, k 517": ((INT8, 1024, 768, 517, None, None, 33), _line(*EXCHANGE(4), 4, 12, 5, 1, 20, 576)),
    "test 96 -> 256, k 300": ((INT8, 256, 96, 300, None, None, 132), _line(*PAIRS, 1, 2, 2, 1, 4, 320)),
    "test 1024 -> 4096, k 260": ((INT8, 4096, 1024, 260, None, None, 8), _line(*PAIRS, 16, 16, 2, 2, 4, 320)),
    "test 8 -> 64, k 1": ((INT8, 64, 8, 1, None, None, 132), _line(*PAIRS, 1, 1, 1, 1, 2, 320)),
    "test 72 -> 320, k 129": ((INT8, 320, 72, 129, None, None, 66), _line(*EXCHANGE(2), 2, 2, 2, 1, 4, 576)),
    "test 40 -> 448, k 257": ((INT8, 448, 40, 257, None, None, 66), _line(*EXCHANGE(2), 2, 1, 3, 1, 6, 576)),
    "test 64 -> 2048, k 9000": ((INT8, 2048, 64, 9000, None, None, 15), _line(*EXCHANGE(8), 8, 1, 71, 1, 120, 576)),
    "test 48 -> 1280, k 7000": ((INT8, 1280, 48, 7000, None, None, 24), _line(*EXCHANGE(5), 5, 1, 55, 1, 120, 576)),
    "test 32 -> 512, k 40000": ((INT8, 512, 32, 40000, None, None, 66), _line(*EXCHANGE(2), 2, 1, 313, 1, 132, 576)),
    # the switches
    "fp16 768 -> 1024, SCONE_FOLD_2SM=0": ((FP16, 1024, 768, K_BENCH, "0", None, 33), _line(*PAIRS, 4, 12, 1024, 1, 148, 320)),
    "int4 1024 -> 4096, SCONE_FOLD_2SM=1": ((INT4, 4096, 1024, K_BENCH, "1", None, 33), _line(*PAIR_TILE, 16, 16, 1024, 1, 148, 320)),
    "int8 768 -> 1024, SCONE_FOLD_XCH=0": ((INT8, 1024, 768, K_BENCH, None, "0", 33), _line(*PAIRS, 4, 12, 1024, 2, 148, 320)),
    # the exchange wins over a forced pair tile, which still applies once the exchange is off
    "int8 768 -> 1024, SCONE_FOLD_2SM=1": ((INT8, 1024, 768, K_BENCH, "1", None, 33), _line(*EXCHANGE(4), 4, 12, 2048, 1, 132, 576)),
    "int8 768 -> 1024, SCONE_FOLD_2SM=1 SCONE_FOLD_XCH=0": ((INT8, 1024, 768, K_BENCH, "1", "0", 33),
                                                           _line(*PAIR_TILE, 4, 12, 1024, 2, 148, 320)),
    # INT8 rows of one chunk need neither the exchange nor a second sweep
    "int8 384 -> 256": ((INT8, 256, 384, K_BENCH, None, None, 132), _line(*PAIRS, 1, 6, 1024, 1, 148, 320)),
    # no exchange cluster fits the device: two sweeps
    "int8 768 -> 1024, no exchange cluster resident": ((INT8, 1024, 768, K_BENCH, None, None, 0), _line(*PAIRS, 4, 12, 1024, 2, 148, 320)),
}


def test_plan_of_the_named_shapes(plan):
    got = plan([case for case, _ in NAMED.values()])
    for (name, (_, want)), line in zip(NAMED.items(), got):
        assert line == want, name


def _fields(line):
    w = line.split()
    return w[0], {k: int(v) for k, v in zip(w[1::2], w[2::2])}


def test_plan_invariants_over_a_grid_of_calls(plan):
    switches = (None, "0", "1")
    for sms in (148, 132, 7):
        cases = [c for c in itertools.product((FP16, INT8, INT4, FP32), range(64, 16385, 64), (8, 384, 512, 1024), (1, 129, 262144, 2**31 - 1),
                                              switches, switches, (0, 1, 15, 33))
                 if c[6] * min((c[1] + 255) // 256, 8) <= sms]  # a device hosts no more exchange clusters than it has SMs for
        seen = set()
        for (quant, H, K, k, sm2, xch, res), line in zip(cases, plan(cases, sms)):
            path, f = _fields(line)
            seen.add(path)
            n = (H + 255) // 256
            assert f["n_chunks"] == n and f["k_blocks"] == (K + 63) // 64, line
            assert f["threads"] == 64 + 32 * f["epi"], line
            assert f["stages"] * f["stage_bytes"] == 4 * 48 * 1024, line
            assert f["grid"] % f["cluster"] == 0 and 0 < f["grid"] <= sms and f["grid"] // f["cluster"] <= f["m_groups"], line
            assert f["m_groups"] == -(-k // (128 * f["tiles"])), line
            exchange = quant == INT8 and 2 <= n <= 8 and res > 0 and xch != "0"
            assert (path == "exchange") == exchange, line
            if exchange:
                assert f["cluster"] == n and f["grid"] == min(res, f["m_groups"]) * n, line
            assert f["sweeps"] == (2 if quant == INT8 and n > 1 and not exchange else 1), line
            if path == "pairtile":
                assert not exchange and (sm2 == "1" or (sm2 is None and quant == FP16 and K >= 512)), line
        assert seen == {"single", "pairs", "pairtile", "exchange"}
