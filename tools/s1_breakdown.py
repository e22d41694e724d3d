# Per-kernel / per-query breakdown of Stage 1 on a synthetic corpus (development tool; needs a GPU).
#   IFX_DBG_DOCS, IFX_DBG_MULTI, IFX_DBG_NQ select the corpus; IFX_LIB an alternative build of libinfidex_gpu.so
import sys, os, ctypes as C
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import infidex_b200 as ib
from infidex_b200 import synth
ND = int(os.environ.get("IFX_DBG_DOCS", "1000000")); MULTI = os.environ.get("IFX_DBG_MULTI", "0") == "1"; NQ = int(os.environ.get("IFX_DBG_NQ", "1000"))
vocab = synth.make_vocab(400_000); docs = synth.gen_docs(ND, vocab, with_description=MULTI); qs = synth.gen_queries(NQ, docs, vocab)
schema, cols = synth.schema_and_columns(docs, MULTI)
e = ib.SearchEngine.CreateDefault(_gpu_lib=os.environ.get('IFX_LIB')); e.IndexColumns(docs["keys"], schema, cols)
h = e.UploadBatch([ib.Query(q, 10) for q in qs])
for r in range(3): e.FlushL2(); st = e.RunBatch(h)
print({k: round(v, 2) if isinstance(v, float) else v for k, v in st.as_dict().items()})
dbg = np.zeros((NQ, 24), np.int64); e._gpu.ifx_debug_stage1_queries(h, dbg.ctypes.data_as(C.c_void_p))
np.save(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "qdbg2_%d.npy" % ND), dbg)
k1 = dbg[:, 4] / 1e6; k2 = dbg[:, 10] / 1e6; mode = dbg[:, 6]; nch = dbg[:, 7]; mx = dbg[:, 8]; ta = dbg[:, 9]; nc = dbg[:, 0]; path = dbg[:, 3]
light = (mx <= 256) & (ta <= 48) & (ta * ((mx + 15) // 16 * 16) <= 6144) & (nc > 0)
print("K1 (select+lookup) sum %.0f ms over queries; selection part %.0f ms; by lookup mode: forward n=%d sum %.0f ms, stream n=%d sum %.0f ms" % (k1.sum(), dbg[:, 2].clip(0).sum() / 1e6, (mode == 1).sum(), k1[mode == 1].sum(), (mode == 2).sum(), k1[mode == 2].sum()))
print("K2 light n=%d sum %.0f ms (mean %.3f ms, max %.2f); heavy n=%d sum %.0f ms (mean %.3f, max %.2f)" % (light.sum(), k2[light].sum(), k2[light].mean() if light.any() else 0, k2[light].max() if light.any() else 0, (~light & (nc > 0)).sum(), k2[~light].sum(), k2[~light & (nc > 0)].mean(), k2[~light].max()))
for name, sel in (("forward", mode == 1), ("stream", mode == 2)):
    if sel.any(): print(name, "mean cand %d mean chunks %.0f mean Ta %.1f mean K1 %.2f ms; lookup part (K1 - selection) mean %.2f ms" % (nc[sel].mean(), nch[sel].mean(), ta[sel].mean(), k1[sel].mean(), (k1[sel] - dbg[sel, 2].clip(0) / 1e6).mean()))
order = np.argsort(-k1)
for i in order[:8]: print("%-36s cand=%7d T=%3d path=%d mode=%d chunks=%4d maxcnt=%4d sel=%.2f K1=%.2f K2=%.2f ms" % (qs[i][:36], nc[i], ta[i], path[i], mode[i], nch[i], mx[i], dbg[i, 2] / 1e6, k1[i], k2[i]))
order = np.argsort(-k2)
for i in order[:5]: print("K2 top: %-30s cand=%7d T=%3d chunks=%4d maxcnt=%4d light=%d K2=%.2f ms" % (qs[i][:30], nc[i], ta[i], nch[i], mx[i], light[i], k2[i]))

if dbg[:, 11:18].sum() > 0:
    for name, sel in (("forward", mode == 1), ("stream", mode == 2)):
        if sel.any(): print(name, "lookup phases, mean kcycles [count+expand, lengths, chunk table+zero, forward-index lookups, clear, list ranges, streamed lookups]:", (dbg[sel, 11:18].mean(0) / 1e3).astype(int), "| selection sticks [sort, tier0/unions, tier1, -]:", (dbg[sel, 20:24].mean(0) / 1e3).astype(int))
