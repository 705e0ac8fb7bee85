"""Workload for compute-sanitizer (memcheck / racecheck / synccheck): every kernel shape on small inputs."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import scone_b200 as sb  # noqa: E402
from scone_b200.utils import synthetic as S  # noqa: E402

cases = [("int8", 1024, 4, 300), ("int4", 512, 5, 70000), ("fp16", 128, 3, 300), ("int4", 4096, 5, 70000), ("fp16", 8192, 2, 300),
         ("int8", 16384, 3, 300), ("fp32", 768, 3, 300)]
for pipe in ("0", "1"):                       # the plain path through the single-ring kernel, then through the three-role pipeline kernel (extra rows always take the pipeline)
  os.environ["SCONE_EMBED_PIPE"] = pipe
  for quant, D, max_n, V in cases:
      toks, lens = S.make_vocab_numpy(1500, max_n, V, seed=1, min_n=1 if max_n < 3 else 2)
      ix = sb.FGramIndex(torch.from_numpy(toks).cuda(), torch.from_numpy(lens).cuda())
      t = sb.CacheTable(1500, D, quant)
      t.store(torch.from_numpy(S.make_rows_numpy(1500, D)).cuda())
      base = torch.randn(V if V < 1000 else 1000, D, device="cuda").to(torch.bfloat16)
      q = torch.from_numpy(S.make_stream_numpy(toks, lens, 3, 130, base.shape[0])).cuda()
      pos = torch.randn(130, D, device="cuda").to(torch.bfloat16)
      out, fid, ml = sb.embed_forward(ix, t, base, q)
      outp, _, _ = sb.embed_forward(ix, t, base, q, pos_emb=pos)
      outa, _, _ = sb.embed_forward(ix, t, base, q, combine="add")
      outap, _, _ = sb.embed_forward(ix, t, base, q, pos_emb=pos, combine="add")
      g = sb.embed_gather(t, base, q, fid)
      m = sb.embed_mean_forward(ix, t, q)
      a = ix.match_all(q)
      torch.cuda.synchronize()
      assert torch.equal(out, g)
      for _ in range(3):                      # back-to-back early-start launches (programmatic dependent launch overlap)
          o2, f2, _ = sb.embed_forward(ix, t, base, q, inputs_stable=True)
      torch.cuda.synchronize()
      assert torch.equal(o2, out) and torch.equal(f2, fid)
      print("ok", "pipe" if pipe == "1" else "bulk", quant, D, max_n, ix.slot_format, flush=True)
os.environ.pop("SCONE_EMBED_PIPE", None)
# a batch large enough for the Bloom pre-filter and the matcher stagger (>= 16 384 positions, >= 2 tiles per matcher)
toks, lens = S.make_vocab_numpy(20000, 4, 5000, seed=3, min_n=2)
ix = sb.FGramIndex(torch.from_numpy(toks).cuda(), torch.from_numpy(lens).cuda())
assert ix.filter_bytes > 0
t = sb.CacheTable(20000, 256, "int8")
t.store(torch.from_numpy(S.make_rows_numpy(20000, 256)).cuda())
base = torch.randn(5000, 256, device="cuda").to(torch.bfloat16)
q = torch.from_numpy(S.make_stream_numpy(toks, lens, 48, 1024, 5000)).cuda()
out, fid, ml = sb.embed_forward(ix, t, base, q)
fid2, ml2 = ix.lookup(q)
torch.cuda.synchronize()
assert torch.equal(fid, fid2) and torch.equal(ml, ml2) and torch.equal(out, sb.embed_gather(t, base, q, fid))
print("ok large batch (pre-filter + stagger)", flush=True)
if os.environ.get("SANITIZE_BUILDERS", "1") == "1":
    # the builders: projection fold (tcgen05 / TMEM / TMA) and vocabulary construction
    for quant in ("fp32", "fp16", "int8", "int4"):
        tq = sb.CacheTable(300, 512, quant)
        tq.store_projected(torch.randn(300, 128, device="cuda"), torch.randn(512, 128, device="cuda"))
    torch.cuda.synchronize()
    print("ok fold", flush=True)
    ex = sb.NGramExtractor(3, 2, 500).fit_device([[1, 2, 3, 4, 1, 2, 3] * 20, [2, 3, 4, 5] * 30, [1, 2, 9] * 10], verbose=False)
    print("ok fit", len(ex), flush=True)
    th = sb.CacheTable(1000, 256, "int8", tier="host")
    th.storage[:10].fill_(1)
    print("ok host alloc", flush=True)
print("sanitizer workload done")
