"""Stage-1 tf lookups streamed container by container: parity with the oracle on corpora of several 65 536-document containers,
with the lookup mode forced to streaming (IFX_S1_LOOKUP=2), forced to the forward index (1: the LD1 unions are still streamed)
and left to the cost model. On the CPU through the kernel emulation, on the GPU through the CUDA library."""
import numpy as np
import pytest

import infidex_b200 as ib
from oracle.oracle import Field as OField
from oracle.oracle import OracleEngine
from parity_util import compare_search, compare_stage1, emu_lib

CONT = 65536


def corpus(n, seed=11):
    """Filler documents of three random words (the synthetic vocabulary has no q, x or y) plus marker words made of those letters:
      zqxjv  every 7th document of the even containers: more than 4096 candidates in a container (sub-chunks), none in the odd ones
      wvyqk  every 11th document of the even containers: `zqxjv wvyqk` takes the AND path and leaves the odd containers empty
      kpfhy  about 400 documents over all containers: a list below 512 postings (no skip table)
    Queries with zqxjw / kpfhq (not in the dictionary, edit distance 1) score LD1 unions from the fuzzy pool."""
    from infidex_b200 import synth
    words = synth.make_vocab(3000)["words"]
    rng = np.random.default_rng(seed)
    pick = rng.integers(0, len(words), (n, 3))
    rare = max(1, n // 400)
    titles = []
    for i in range(n):
        t = [words[pick[i, 0]], words[pick[i, 1]], words[pick[i, 2]]]
        even = (i // CONT) % 2 == 0
        if even and i % 7 == 0:
            t.append("zqxjv")
        if even and i % 11 == 0:
            t.append("wvyqk")
        if i % rare == 3:
            t.append("kpfhy")
        titles.append(" ".join(t))
    qs = ["zqxjv wvyqk", "zqxjv", "wvyqk", "kpfhy", "kpfhy zqxjv", "kpfhy wvyqk", "zqxjw", "zqxjw wvyqk", "kpfhq", "kpfhq zqxjv",
          "zqxjw kpfhy", " ".join(titles[5][:2]), titles[12], titles[70001].split()[0] + " zqxjv", titles[3].split()[1] + " kpfhy"]
    return titles, qs


def _pair(titles, gpu_lib=None):
    keys = np.arange(len(titles), dtype=np.int64)
    eng = ib.SearchEngine(_gpu_lib=gpu_lib) if gpu_lib else ib.SearchEngine.CreateDefault()
    eng.IndexColumns(keys, [ib.Field("content")], [titles])
    orc = OracleEngine([OField("content", ib.Weight.Med, True, False, False)])
    orc.index_columns(keys, [titles])
    return eng, orc


@pytest.fixture(scope="module")
def emu_pair():
    titles, qs = corpus(4 * CONT + 40_000)      # five containers, the last one partial
    eng, orc = _pair(titles, gpu_lib=emu_lib())
    return eng, orc, qs


@pytest.mark.parametrize("mode", [None, "1", "2"])
def test_emu_lookup_containers(emu_pair, mode, monkeypatch):
    eng, orc, qs = emu_pair
    if mode is None:
        monkeypatch.delenv("IFX_S1_LOOKUP", raising=False)
    else:
        monkeypatch.setenv("IFX_S1_LOOKUP", mode)
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs)


@pytest.fixture(scope="module")
def gpu_pair():
    titles, qs = corpus(1_200_000)      # 19 containers
    eng, orc = _pair(titles)
    return eng, orc, qs


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [None, "1", "2"])
def test_gpu_lookup_containers(gpu_pair, mode, monkeypatch):
    eng, orc, qs = gpu_pair
    if mode is None:
        monkeypatch.delenv("IFX_S1_LOOKUP", raising=False)
    else:
        monkeypatch.setenv("IFX_S1_LOOKUP", mode)
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs)
