"""CPU: trigram scores from the language model laid out as arrays (integration/ps_search_cuda.c:
cuda_ngram_export_lm; scoring restated in oracle/ps_oracle.c:lmarr_tg and, for the device, in
pocketsphinx_b200/csrc/psb_lm_core.h) against the reference's own ngram_tg_score: a committed sample for
the turtle LM, and live -- every (w, h1, h2) of the turtle and tidigits vocabularies, and every existing
bigram / trigram entry plus random queries of the 72 k-word en-us LM (whose trie contains unsorted ranges:
the search has to be the reference's own interpolation search, a binary search disagrees)."""
import os

import numpy as np
import pytest

from conftest import golden
from oracle import oracle, refdrv


def test_array_lm_scores_match_committed_reference_sample():
    g = golden("en_us_fwdtree.npz")
    assert np.array_equal(oracle.lm_scores(g["lmarr"], g["lmarr_queries"]), g["lmarr_scores"])


live = pytest.mark.skipif(not refdrv.available(), reason="oracle/_ref/libpsref.so not built")
REF = os.path.dirname(refdrv.LIB_PATH)


def _all_queries(nw):
    hs = np.arange(-1, nw)
    return np.array([(w, h1, h2) for w in range(nw) for h1 in hs for h2 in hs], np.int32)


@live
@pytest.mark.parametrize("which", ["turtle", "tidigits"])
def test_every_triple_of_the_small_lms(which):
    hd, lm, dic = {"turtle": (os.path.join(REF, "model", "en-us"), os.path.join(REF, "data", "turtle.lm.bin"),
                              os.path.join(REF, "data", "turtle.dic")),
                   "tidigits": (os.path.join(REF, "model", "tidigits_hmm"), os.path.join(REF, "model", "tidigits_lm", "tidigits.lm.bin"),
                                os.path.join(REF, "model", "tidigits_lm", "tidigits.dic"))}[which]
    arr, _ = refdrv.lm_arrays(hd, lm, dic)
    q = _all_queries(int(arr[7]))
    arr, want = refdrv.lm_arrays(hd, lm, dic, q)
    assert np.array_equal(oracle.lm_scores(arr, q), want)


BIG_LM = os.path.join(REF, "model", "en-us.lm.bin")


@live
@pytest.mark.skipif(not os.path.exists(BIG_LM), reason="oracle/_ref/model/en-us.lm.bin not built")
def test_en_us_lm_existing_ngrams_and_random_queries():
    hd, dic = os.path.join(REF, "model", "en-us"), os.path.join(REF, "model", "cmudict-en-us.dict")
    arr, _ = refdrv.lm_arrays(hd, BIG_LM, dic)
    order, V, n2, n3 = (int(x) for x in arr[:4])
    nw = int(arr[7])
    assert order == 3 and V > 70000
    rng = np.random.default_rng(0)
    widmap = arr[10:10 + nw]
    inlm = np.nonzero(widmap >= 0)[0]
    o = 10 + nw
    uni_next = arr[o + 2 * V:o + 3 * V + 1]
    o2 = o + 3 * V + 1
    bg_word, bg_next = arr[o2:o2 + n2], arr[o2 + 3 * n2:o2 + 4 * n2 + 1]
    tg_word = arr[o2 + 4 * n2 + 1:o2 + 4 * n2 + 1 + n3]
    inv = np.full(V, -1, np.int64)
    inv[widmap[inlm]] = inlm
    n2u = int(uni_next[V])
    n3u = int(bg_next[n2u])
    ti = np.arange(0, n3u, 3)                                    # every third trigram entry, every fifth bigram entry
    b_of_t = np.searchsorted(bg_next[:n2u + 1], ti, side="right") - 1
    w_of_t = np.searchsorted(uni_next, b_of_t, side="right") - 1
    q4 = np.stack([inv[w_of_t], inv[bg_word[b_of_t]], inv[tg_word[ti]]], 1)
    bi = np.arange(0, n2u, 5)
    w_of_b = np.searchsorted(uni_next, bi, side="right") - 1
    q3 = np.stack([inv[w_of_b], inv[bg_word[bi]], rng.choice(inlm, len(bi))], 1)
    q1 = np.stack([rng.choice(inlm, 200000), rng.choice(inlm, 200000), rng.choice(inlm, 200000)], 1)
    q = np.concatenate([q1, q3, q4]).astype(np.int32)
    q = q[(q >= -1).all(1) & (q[:, 0] >= 0)]
    arr, want = refdrv.lm_arrays(hd, BIG_LM, dic, q)
    assert np.array_equal(oracle.lm_scores(arr, q), want)
    # the trie is not sorted everywhere: that is why the search has to be the reference's own
    d = np.diff(tg_word[:n3u].astype(np.int64))
    inside = np.ones(len(d), bool)
    inside[bg_next[1:n2u][(bg_next[1:n2u] > 0) & (bg_next[1:n2u] < n3u)] - 1] = False      # differences across range boundaries
    assert (d[inside] <= 0).sum() > 0
