"""The f-gram index's plan (scone_b200/csrc/index_plan.h), compiled on the host with g++.

The plan alone decides the slot format, the capacity and the pre-filter size scone_index_create gives a vocabulary; these
tests pin those decisions at the formats' limits, for the two test switches and for the load factors and vocabulary sizes
the GPU tests and the benchmark use.
"""

import pytest

from plan_driver import PlanDriver


@pytest.fixture(scope="module")
def plan(tmp_path_factory):
    """plan(cases) -> (format name, slot bytes, cap, filter words, filter_always, format number) per case; a case is
    (n, max_n, largest token, load factor, SCONE_INDEX_FORMAT, SCONE_INDEX_FILTER)."""
    try:
        driver = PlanDriver.build(str(tmp_path_factory.mktemp("index_plan")))
    except FileNotFoundError:
        pytest.skip("no host C++ compiler")

    def run(cases):
        out = []
        for line in driver.index(cases):
            w = line.split()
            f = dict(zip(w[1::2], (int(x) for x in w[2::2])))
            out.append((w[0], f["slot_bytes"], f["cap"], f["filter_words"], f["filter_always"], f["format"]))
        return out
    return run


def _formats(plan, cases):
    return [p[0] for p in plan(cases)]


def test_format_at_the_token_and_length_limits(plan):
    # (n, max_n, largest token) -> format: compact-16 holds six tokens < 65535, compact-20 five tokens < 1048575 and fewer
    # than 2^28 - 1 f-grams, 32-byte slots everything else
    want = {
        (1000, 5, 65534): "compact16",
        (1000, 5, 65535): "compact20",
        (1000, 5, 1048574): "compact20",
        (1000, 5, 1048575): "wide32",
        (1000, 5, 2**31 - 1): "wide32",
        (1000, 6, 100): "compact16",
        (1000, 6, 65535): "wide32",
        (1000, 7, 100): "wide32",
        (1000, 1, 0): "compact16",
        (0, 3, 0): "compact16",
        (2**28 - 2, 5, 70000): "compact20",
        (2**28 - 1, 5, 70000): "wide32",
        (2**28 - 1, 5, 100): "compact16",
        (2**31 - 2, 6, 65534): "compact16",
    }
    got = plan([(n, m, t, 0.0, None, None) for n, m, t in want])
    assert [g[0] for g in got] == list(want.values())
    assert all(g[1] == (32 if g[0] == "wide32" else 16) for g in got)


def test_format_names_match_the_python_binding(plan):
    """scone_b200.index names scone_index_info's slot_format by its own copy of the rows' names: the two must agree."""
    from scone_b200.index import SLOT_FORMATS
    got = plan([(1000, 5, 100, 0.0, "wide", None), (1000, 5, 100, 0.0, None, None), (1000, 5, 70000, 0.0, None, None)])
    assert {g[5]: g[0] for g in got} == dict(enumerate(SLOT_FORMATS))


def test_format_switches(plan):
    vocabularies = [(1000, 5, 100), (1000, 6, 100), (1000, 5, 70000), (1000, 5, 1048575), (2**28 - 1, 5, 70000)]
    auto = ["compact16", "compact16", "compact20", "wide32", "wide32"]
    cases = lambda env: [(n, m, t, 0.0, env, None) for n, m, t in vocabularies]
    assert _formats(plan, cases(None)) == auto
    assert _formats(plan, cases("wide")) == ["wide32"] * 5
    # compact-20 wherever it fits, the automatic choice where it does not
    assert _formats(plan, cases("prefer-compact20")) == ["compact20", "compact16", "compact20", "wide32", "wide32"]
    # any other value is the automatic choice, the names of the formats included
    for other in ("compact", "compact20", "compact16", "WIDE"):
        assert _formats(plan, cases(other)) == auto, other


def test_capacity_from_the_load_factor(plan):
    # (n, load factor) -> slots: n / lf + 1, at least 64, rounded up to a multiple of 4; lf <= 0 means 0.25
    want = {
        (1000, 0.0): 4004, (1000, -1.0): 4004, (1000, 0.25): 4004, (1000, 0.5): 2004, (1000, 0.9): 1112,
        (0, 0.0): 64, (10, 0.9): 64, (15, 0.25): 64, (16, 0.25): 68, (50_000, 0.0): 200_004, (10_000_000, 0.0): 40_000_004,
        (33, 0.5): 68, (3, 0.1): 64, (7, 0.1): 72,
    }
    got = plan([(n, 5, 100, lf, None, None) for n, lf in want])
    assert [g[2] for g in got] == list(want.values())


def test_filter_size(plan):
    # (n, SCONE_INDEX_FILTER) -> (filter words, filter_always): 16 bits per f-gram up to 12 M f-grams, 8 bits up to 48 M,
    # none above; at least 1024 words, a multiple of 32
    want = {
        (0, None): (0, 0), (0, "always"): (0, 0),
        (1, None): (1024, 0),
        (2047, None): (1024, 0), (2049, None): (1025 + 31 & ~31, 0),
        (50_000, None): (25_024, 0),                         # test_prefilter_never_changes_a_result's 4 * ((N + 1) // 2 + 31) // 32 * 32 bytes
        (10_000_000, None): (5_000_000, 0),                  # config 3: a 20 MB filter
        (12_000_000, None): (6_000_000, 0), (12_000_001, None): (3_000_032, 0),
        (48_000_000, None): (12_000_000, 0), (48_000_001, None): (0, 0),
        (48_000_001, "always"): (12_000_032, 1), (2**31 - 2, "always"): ((2**31 - 2 + 3) // 4 + 31 & ~31, 1),
        (50_000, "never"): (0, 0), (1, "never"): (0, 0), (50_000, "always"): (25_024, 1), (50_000, "sometimes"): (25_024, 0),
    }
    got = plan([(n, 5, 100, 0.0, None, env) for n, env in want])
    assert [(g[3], g[4]) for g in got] == list(want.values())
