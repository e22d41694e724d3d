"""CPU-side logic tests: the kernel sources compiled as a single-threaded host emulation (tests/emu) against the oracle.
This checks the *logic* of the device code without a GPU; the real parity tests are the `-m gpu` ones."""
import numpy as np
import pytest

import infidex_b200 as ib
from conftest import REFERENCE_10
from infidex_b200 import synth
from oracle.oracle import OracleEngine
from parity_util import build_pair, compare_search, compare_stage1, emu_lib


@pytest.fixture(scope="module")
def emu():
    return emu_lib()


def test_emu_reference_corpus(emu):
    eng = ib.SearchEngine(_gpu_lib=emu)
    eng.IndexDocuments([ib.Document(i + 1, t) for i, t in enumerate(REFERENCE_10)])
    orc = OracleEngine(); orc.index_texts(REFERENCE_10, keys=np.arange(1, 11))
    qs = ["batman", "qick fux", "battamam", "new york", "speeding", "quik fox", "the", "fox", "gotham cty", "a", "wonder woman protects", ""]
    assert not compare_search(eng, orc, qs)
    assert not compare_stage1(eng, orc, qs)


def test_emu_movies(emu, movie_titles, oracle_movies):
    eng = ib.SearchEngine(_gpu_lib=emu)
    eng.IndexColumns(np.arange(len(movie_titles)), [ib.Field("content")], [movie_titles])
    qs = ["redemption sh", "Shaaawshank", "the amtrix", "star", "fellowship of the ring", "te matri", "san a", "the", "new york", "x-men", "Música"]
    assert not compare_stage1(eng, oracle_movies, qs)
    assert not compare_search(eng, oracle_movies, qs)


@pytest.mark.parametrize("multi", [False, True])
def test_emu_synthetic(emu, multi):
    vocab = synth.make_vocab(30_000)
    docs = synth.gen_docs(30_000 if not multi else 15_000, vocab, with_description=multi)
    qs = synth.gen_queries(150, docs, vocab)
    schema, cols = synth.schema_and_columns(docs, multi)
    eng, orc = build_pair(docs["keys"], schema, cols, gpu_lib=emu)
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs)
    # the split form (upload, run, read back) returns the records ifx_search_batch just returned for the same batch
    h = eng.UploadBatch([ib.Query(q, 10) for q in qs]); eng.RunBatch(h); got = eng.DownloadBatch(h, len(qs), 10); eng.FreeBatch(h)
    want = dict(zip(("doc_key", "score", "tie", "n", "total_candidates", "status"), eng.last_raw))
    assert all(np.array_equal(got[k], want[k]) for k in ("n", "total_candidates", "status"))
    assert all(np.array_equal(got[k][i, :n], want[k][i, :n]) for k in ("doc_key", "score", "tie") for i, n in enumerate(want["n"]))     # slots after n are undefined
    if multi:
        flt = ib.Filter.Parse("year >= 2000 AND rating > 7.0")
        assert not compare_search(eng, orc, qs[:80], flt=flt, facets=True)


def test_emu_ld1_more_than_1024_matches(emu):
    """An unknown word with > 1024 dictionary terms at edit distance 1: the reference keeps the first 1024 in trie (ordinal) order
    (VectorModel.cs:662); the unordered fast scan must fall back to the ordered one."""
    alpha = [chr(c) for c in range(0x4E00, 0x4E00 + 330)]          # 330 distinct letters
    words = [a + "bcd" for a in alpha] + ["a" + a + "cd" for a in alpha] + ["ab" + a + "d" for a in alpha] + ["abc" + a for a in alpha]
    titles = [w + " filler%d" % (i % 7) for i, w in enumerate(words)]
    eng = ib.SearchEngine(_gpu_lib=emu); eng.IndexColumns(np.arange(len(titles)), [ib.Field("content")], [titles])
    orc = OracleEngine(); orc.index_texts(titles, keys=np.arange(len(titles)))
    qs = ["abcd", "abcd filler3", "xbcd"]
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs)


def test_emu_dense_terms_and_full_chunks(emu):
    """Few distinct words over many docs: every list is dense (bitmap AND tiers, bitset-mode intersections), chunks are full
    (4096 candidates, > 512 flush survivors while the heap fills, ties at the threshold)."""
    rng = np.random.Generator(np.random.PCG64(7))
    vocab = ["alpha", "alphabet", "beta", "betamax", "gamma", "gammas", "delta", "deltas", "omega", "omegas", "sigma", "sigmas"]
    n = 40_000
    titles = [" ".join(vocab[j] for j in rng.integers(0, len(vocab), int(rng.integers(1, 5)))) for _ in range(n)]
    eng = ib.SearchEngine(_gpu_lib=emu); eng.IndexColumns(np.arange(n), [ib.Field("content")], [titles])
    orc = OracleEngine(); orc.index_texts(titles, keys=np.arange(n))
    qs = ["alpha beta", "alphabet gamma delta", "omegas sigma", "gama", "betamax alpha omega sigma", "delt sigm", "alpha"]
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs)


def test_emu_query_parameter_edges(emu, movie_titles, oracle_movies):
    """Result limits and depths of QueryTests.cs (1, 3, more than there are matches), coverage off, very long / degenerate queries."""
    eng = ib.SearchEngine(_gpu_lib=emu)
    eng.IndexColumns(np.arange(len(movie_titles)), [ib.Field("content")], [movie_titles])
    qs = ["star wars", "the lord of the rings", "godfather", "zzzzqqqq", "   ", "", "matrix reloaded revolutions", "q" * 60, "love " * 40]
    for mr, depth in ((1, 500), (3, 50), (1000, 500), (10, 10)):
        assert not compare_search(eng, oracle_movies, qs, max_results=mr, depth=depth), (mr, depth)
    assert not compare_search(eng, oracle_movies, qs, coverage=False)
    assert not compare_stage1(eng, oracle_movies, qs, depth=64)
    # beyond the fixed query buffer (256 UTF-16 units) the product must say so instead of answering something else
    r = eng.SearchBatch([ib.Query("a" * 300, 10)])[0]
    assert r.Status & 4 and not r.Records


def test_emu_small_reference_corpora(emu):
    """The small corpora of SearchEngineTests.cs / QueryTests.cs, including twenty identical documents (every score ties; only the
    heap layout and the key order decide who survives) -- product logic against the oracle, bit for bit."""
    corpora = [
        (["hello world", "goodbye world", "hello there"], 1, ["hello world", "hello", "wrld", "goodby"]),
        (["batman and robin", "superman flies high", "spiderman swings"], 1, ["batmam", "superman", "swings high"]),
        (["the quick brown fox", "the lazy brown dog", "a quick decision", "quick brown"], 1, ["quick brown", "brown", "quick decision"]),
        (["batman saves the day"] * 20, 0, ["batman", "saves the day", "batmen"]),
        (["batman saves the day story %d" % i for i in range(20)], 0, ["batman", "story 7", "day story"]),
    ]
    for texts, k0, qs in corpora:
        keys = np.arange(k0, k0 + len(texts))
        eng = ib.SearchEngine(_gpu_lib=emu); eng.IndexColumns(keys, [ib.Field("content")], [texts])
        orc = OracleEngine(); orc.index_texts(texts, keys=keys)
        for mr in (5, 8, 10):
            assert not compare_search(eng, orc, qs, max_results=mr), (texts[0], mr)
        assert not compare_stage1(eng, orc, qs)


def test_concurrent_search_calls_are_serialised_correctly(emu, movie_titles):
    """ThreadSafetyTests.cs in spirit: many threads call Search on one engine (readers under the C# read lock); the C-ABI serialises
    the calls on its single batch workspace and every caller must get exactly its own answer."""
    import threading
    eng = ib.SearchEngine(_gpu_lib=emu)
    eng.IndexColumns(np.arange(5000), [ib.Field("content")], [movie_titles[:5000]])
    qs = ["star wars", "the matrix", "godfather", "lord rings", "toy story", "batman", "alien", "love", "night", "dark knight"]
    want = {q: [(e.DocumentId, e.Score, e.Tiebreaker) for e in eng.Search(ib.Query(q, 10)).Records] for q in qs}
    errors = []

    def worker(k):
        try:
            for i in range(30):
                q = qs[(i * 7 + k) % len(qs)]
                got = [(e.DocumentId, e.Score, e.Tiebreaker) for e in eng.Search(ib.Query(q, 10)).Records]
                if got != want[q]:
                    errors.append((k, q))
        except Exception as e:      # noqa: BLE001
            errors.append((k, repr(e)))
    ts = [threading.Thread(target=worker, args=(k,)) for k in range(6)]
    [t.start() for t in ts]; [t.join() for t in ts]
    assert not errors, errors[:3]


def test_emu_several_containers(emu):
    """More than 65 536 documents: container runs, per-container skip-table windows, tail chunks per container, bitset-mode tiers --
    the multi-container control flow on the CPU (the GPU tests repeat it at 300 k documents)."""
    vocab = synth.make_vocab(60_000)
    docs = synth.gen_docs(150_000, vocab)
    qs = synth.gen_queries(50, docs, vocab)
    schema, cols = synth.schema_and_columns(docs, False)
    eng, orc = build_pair(docs["keys"], schema, cols, gpu_lib=emu)
    assert not compare_stage1(eng, orc, qs)
    assert not compare_search(eng, orc, qs[:25])


def test_emu_degenerate_corpora(emu):
    """No documents at all; documents that are empty, blank, delimiter-only or shorter than an n-gram."""
    eng = ib.SearchEngine(_gpu_lib=emu); eng.IndexColumns(np.zeros(0, np.int64), [ib.Field("content")], [[]])
    r = eng.Search(ib.Query("hello", 10)); assert not r.Records and not (r.Status & ~8)
    texts = ["", "   ", "a", "ab", "---", "hello"]
    eng = ib.SearchEngine(_gpu_lib=emu); eng.IndexColumns(np.arange(len(texts)), [ib.Field("content")], [texts])
    orc = OracleEngine(); orc.index_texts(texts, keys=np.arange(len(texts)))
    qs = ["hello", "hel", "a", "ab", "---", "x y z", "hellp", "hello hello"]
    assert not compare_search(eng, orc, qs) and not compare_stage1(eng, orc, qs)


def test_emu_short_queries(emu, movie_titles, oracle_movies):
    """Queries without a word of >= 3 characters (SURVEY 8f-1): champion lists, single-character scan, SearchShortQuery with its fuzzy
    fallback -- ids, Score bits and TotalCandidates against the oracle (which the reference's own short-query tests pin)."""
    eng = ib.SearchEngine(_gpu_lib=emu)
    eng.IndexColumns(np.arange(len(movie_titles)), [ib.Field("content")], [movie_titles])
    qs = ["a", "x", "th", "io", "as am", "a b", "é", "of", "I", "to be", "x y z", "q", "zz", "9"]
    for mx in (10, 100):
        bad = compare_search(eng, oracle_movies, qs, max_results=mx)
        assert not bad, (mx, bad[:3])
    for texts in (["a", "b", "ab", "a b", "b a", "c"], ["x", "xx", "x x", "The X", "y"]):       # the reference's tiny short-query corpora in spirit
        from oracle.oracle import OracleEngine
        orc = OracleEngine(); orc.index_texts(texts); e2 = ib.SearchEngine(_gpu_lib=emu); e2.IndexColumns(np.arange(len(texts)), [ib.Field("content")], [texts])
        bad = compare_search(e2, orc, ["a", "b", "x", "ab", "a b", "xx", "y z"], max_results=10)
        assert not bad, bad[:3]
