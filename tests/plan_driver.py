"""Host-side driver of the launch plans of the fused path (scone_b200/csrc/embed_plan.h) and of the projection fold
(fold_plan.h), and of the f-gram index's plan (index_plan.h), compiled with g++.

The plans are plain C++ with no CUDA header, so they run on any host.  Tests use the driver to pin the kernel a call gets
(test_embed_plan.py, test_fold_plan.py), the shape of an index (test_index_plan.py) and to pick, for every kernel the library compiles, a call that launches it
(test_gpu_kernel_matrix.py).  A helper module, not a conftest: importing it does nothing until ``PlanDriver`` is built.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import tempfile
from typing import Iterable, List, Optional, Sequence, Tuple

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scone_b200", "csrc")
FAMILIES = ("bulk", "pipe", "ldg")

# argv: shapes | plan <sms> | detail <sms> | fold <sms> | index.  plan / detail read one call per line:
# D row_stride pos additive resolved P SCONE_EMBED_PIPE(or -) T
# fold reads: quant H K k SCONE_FOLD_2SM(or -) SCONE_FOLD_XCH(or -) resident_exchange_clusters
# and index reads: n max_n max_tok load_factor SCONE_INDEX_FORMAT(or -) SCONE_INDEX_FILTER(or -)
SOURCE = r"""
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "embed_plan.h"
#include "fold_plan.h"
#include "index_plan.h"
using namespace scone;
static int fold(int sms) {
    const char *path[kNumFoldPaths] = {"single", "pairs", "pairtile", "exchange"};
    int quant, H, K, resident;
    long long k;
    char sm2[8], xch[8];
    while (scanf("%d %d %d %lld %7s %7s %d", &quant, &H, &K, &k, sm2, xch, &resident) == 7) {
        const FoldCall c{quant, H, K, k, sms, sm2[0] == '-' ? nullptr : sm2, xch[0] == '-' ? nullptr : xch, resident};
        const FoldPlan pl = plan_fold(c);
        const FoldPathRow &r = kFoldPaths[pl.path];
        printf("%s cluster %d tiles %d epi %d stages %d stage_bytes %d box %d n_chunks %d k_blocks %d m_groups %d sweeps %d grid %d "
               "threads %d\n", path[pl.path], pl.cluster, r.tiles, r.epi_warps, r.stages, r.stage_bytes, r.w_box_rows, pl.n_chunks,
               pl.k_blocks, pl.m_groups, pl.sweeps, pl.grid, pl.threads);
    }
    return 0;
}
static int index() {
    long long n;
    int max_n, max_tok;
    double lf;
    char fmt[32], filt[32];
    while (scanf("%lld %d %d %lf %31s %31s", &n, &max_n, &max_tok, &lf, fmt, filt) == 6) {
        const IndexPlan pl = plan_index(IndexCall{n, max_n, max_tok, lf, fmt[0] == '-' ? nullptr : fmt, filt[0] == '-' ? nullptr : filt});
        printf("%s format %d slot_bytes %d cap %llu filter_words %u filter_always %d\n", kSlotFormats[pl.format].name,
               (int)pl.format, kSlotFormats[pl.format].slot_bytes, (unsigned long long)pl.cap, pl.filter_words, (int)pl.filter_always);
    }
    return 0;
}
int main(int argc, char **argv) {
    const char *fam[3] = {"bulk", "pipe", "ldg"};
    if (argc == 2 && !strcmp(argv[1], "shapes")) {
        for (int r = 0; r < kNumShapes; ++r) {
            const ShapeRow &s = kShapes[r];
            printf("%d %s %d %d %d %d %u %u %d\n", r, fam[s.family], s.nm, s.nl, s.ng, s.minb, s.plain, s.add, (int)s.stagger);
        }
        return 0;
    }
    if (argc == 2 && !strcmp(argv[1], "index")) return index();
    if (argc != 3) return 2;
    if (!strcmp(argv[1], "fold")) return fold(atoi(argv[2]));
    const bool detail = !strcmp(argv[1], "detail");
    const int sms = atoi(argv[2]);
    long long D, rs, T;
    int pos, add, res, P;
    char env[8];
    while (scanf("%lld %lld %d %d %d %d %7s %lld", &D, &rs, &pos, &add, &res, &P, env, &T) == 8) {
        const EmbedCall c{D, rs, pos != 0, add != 0, res != 0, P, env[0] == '-' ? nullptr : env, T, sms};
        const EmbedPlan pl = plan_embed(c);
        const ShapeRow &s = kShapes[pl.row];
        if (detail) {
            const int ring = s.family == kBulk ? pl.bulk.ring : s.family == kPipe ? pl.pipe.ring : 0;
            const int meta = s.family == kPipe ? pl.pipe.meta_ring : 0;
            printf("%d %d %d %lld %lld %d %d %d\n", (int)pl.row, pl.P, (int)pl.add, (long long)pl.num_tiles, (long long)pl.grid, ring,
                   meta, pl.stagger_ns);
            continue;
        }
        printf("%s nm %d nl %d ng %d minb %d budget %d P %d add %d", fam[s.family], s.nm, s.nl, s.ng, s.minb, s.budget, pl.P, (int)pl.add);
        if (s.family == kBulk) printf(" ring %d slot %d", pl.bulk.ring, pl.bulk.slot_bytes);
        if (s.family == kPipe)
            printf(" ring %d meta %d slot %d add_off %d pos_off %d tile %d", pl.pipe.ring, pl.pipe.meta_ring, pl.pipe.slot_bytes,
                   pl.pipe.add_off, pl.pipe.pos_off, pl.pipe.tile_bytes);
        printf(" smem %d stagger %d grid %lld threads %u\n", pl.smem_bytes, pl.stagger_ns, (long long)pl.grid, pl.threads);
    }
}
"""

# (D, row_stride, position rows, additive, resolved ids, P, SCONE_EMBED_PIPE or None, T)
Call = Tuple[int, int, int, int, int, int, Optional[str], int]
# (quant, H, K, k, SCONE_FOLD_2SM or None, SCONE_FOLD_XCH or None, resident exchange clusters)
FoldCall = Tuple[int, int, int, int, Optional[str], Optional[str], int]
# (n, max_n, largest token, load factor, SCONE_INDEX_FORMAT or None, SCONE_INDEX_FILTER or None)
IndexCall = Tuple[int, int, int, float, Optional[str], Optional[str]]


class ShapeRow:
    """One row of kShapes."""

    def __init__(self, line: str):
        w = line.split()
        self.row, self.family = int(w[0]), w[1]
        self.nm, self.nl, self.ng, self.minb, self.plain, self.add, self.stagger = (int(x) for x in w[2:])

    def instances(self) -> List[Tuple[int, int, int]]:
        """The (row, P, ADD) combinations the library compiles for this row."""
        return [(self.row, P, add) for add, mask in ((0, self.plain), (1, self.add)) for P in (1, 2, 4, 8) if mask & P]


class Planned:
    """What plan_embed() returns for one call, as far as the tests need it."""
    __slots__ = ("row", "P", "add", "num_tiles", "grid", "ring", "meta", "stagger")

    def __init__(self, line: str):
        self.row, self.P, self.add, self.num_tiles, self.grid, self.ring, self.meta, self.stagger = (int(x) for x in line.split())

    @property
    def instance(self) -> Tuple[int, int, int]:
        return self.row, self.P, self.add


class PlanDriver:
    """The compiled driver.  ``shapes()`` lists kShapes; ``plan`` / ``detail`` plan a batch of calls for ``sms`` SMs."""

    def __init__(self, exe: str):
        self.exe = exe

    @classmethod
    def build(cls, directory: Optional[str] = None) -> "PlanDriver":
        cxx = shutil.which("g++")
        if cxx is None:
            raise FileNotFoundError("no host C++ compiler (g++)")
        d = directory or tempfile.mkdtemp(prefix="scone_plan_")
        src, exe = os.path.join(d, "plan_driver.cpp"), os.path.join(d, "plan_driver")
        with open(src, "w") as f:
            f.write(SOURCE)
        subprocess.run([cxx, "-std=c++17", "-O2", "-Wall", "-Werror", "-I", CSRC, src, "-o", exe], check=True)
        return cls(exe)

    def _run(self, args: Sequence[str], cases: Iterable[Call]) -> List[str]:
        cases = list(cases)
        return self._lines(args, "".join(f"{D} {rs} {int(pos)} {int(add)} {int(res)} {P} {env or '-'} {T}\n"
                                         for D, rs, pos, add, res, P, env, T in cases), len(cases))

    def _lines(self, args: Sequence[str], text: str, n: int) -> List[str]:
        out = subprocess.run([self.exe, *args], input=text, capture_output=True, text=True, check=True).stdout.splitlines()
        assert len(out) == n
        return out

    def shapes(self) -> List[ShapeRow]:
        out = subprocess.run([self.exe, "shapes"], capture_output=True, text=True, check=True).stdout.splitlines()
        return [ShapeRow(line) for line in out]

    def plan(self, cases: Iterable[Call], sms: int) -> List[str]:
        """One line per call: family, shape, P, ring layout, shared memory, stagger, grid and threads."""
        return self._run(["plan", str(sms)], cases)

    def detail(self, cases: Iterable[Call], sms: int) -> List[Planned]:
        return [Planned(line) for line in self._run(["detail", str(sms)], cases)]

    def fold(self, cases: Iterable[FoldCall], sms: int) -> List[str]:
        """plan_fold() of each call: one line with the path, its row of kFoldPaths and the launch."""
        cases = list(cases)
        return self._lines(["fold", str(sms)], "".join(f"{q} {H} {K} {k} {s or '-'} {x or '-'} {res}\n" for q, H, K, k, s, x, res in cases),
                           len(cases))

    def index(self, cases: Iterable[IndexCall]) -> List[str]:
        """plan_index() of each call: the slot format's name, number and size, the capacity, the filter words and filter_always."""
        cases = list(cases)
        return self._lines(["index"], "".join(f"{n} {m} {t} {lf!r} {f or '-'} {x or '-'}\n" for n, m, t, lf, f, x in cases), len(cases))
