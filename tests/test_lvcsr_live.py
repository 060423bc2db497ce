"""CPU, build container (needs oracle/_ref/libpsref.so AND the reference's en-us.lm.bin): the reference's
own large-vocabulary configuration -- cmudict (134 865 words), the 72 k-word en-us trigram LM -- decoding
goforward.raw: lextree of 723 roots and 152 500 non-root channels exported without a dense LM table, the
LM as arrays.  Both passes of the oracle restatement and of the device search's phase code (host
emulation, both thread orders) must reproduce the reference's backpointer tables entry for entry."""
import os

import numpy as np
import pytest

from oracle import oracle, refdrv
from test_ngf_emul import emuls, run_second  # noqa: F401
from test_ngs_emul import run_emul as run_first

REF = os.path.dirname(refdrv.LIB_PATH)
BIG_LM = os.path.join(REF, "model", "en-us.lm.bin")
pytestmark = [pytest.mark.skipif(not refdrv.available(), reason="oracle/_ref/libpsref.so not built"),
              pytest.mark.skipif(not os.path.exists(BIG_LM), reason="oracle/_ref/model/en-us.lm.bin not built")]


def test_large_vocabulary_decode(emuls):  # noqa: F811
    f1, f2 = emuls
    hd, dic = os.path.join(REF, "model", "en-us"), os.path.join(REF, "model", "cmudict-en-us.dict")
    pcm = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
    ref = refdrv.RefModel(hd)
    pk = ref.packed()
    scr = np.ascontiguousarray(ref.score(ref.featurize_fresh(pcm)))
    ref.close()
    first = refdrv.fwdtree(hd, BIG_LM, dic, pcm, dense_lm=False)
    both = refdrv.fwdtree(hd, BIG_LM, dic, pcm, dense_lm=False, fwdflat="yes")
    assert first["n_words"] > 130000 and first["n_nonroot"] > 100000 and first["n_lm"] == 0 and both["hyp"] == "go forward ten meters"
    lma, _ = refdrv.lm_arrays(hd, BIG_LM, dic)
    nc = first["n_ci"]
    o1 = oracle.fwdtree_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], first["info"], first["model"], scr, lm_arrays=lma)
    assert np.array_equal(o1[0], first["bp"]) and np.array_equal(o1[1], first["bss"]) and np.array_equal(o1[2], first["bp_idx"])
    o2 = oracle.fwdflat_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], pk["phone_ssid"][:nc], both["info"], both["model"], o1[0], scr,
                            lm_arrays=lma)
    assert np.array_equal(o2[0], both["bp"]) and np.array_equal(o2[1], both["bss"]) and np.array_equal(o2[2], both["bp_idx"])
    n1, bp1, bss1, idx1 = run_first(f1, pk, first["info"], first["model"], scr, len(first["bp"]) + 64, len(first["bss"]) + 4096, lm_arrays=lma)
    assert n1 == len(first["bp"]) and np.array_equal(bp1, first["bp"]) and np.array_equal(bss1, first["bss"]) and np.array_equal(idx1, first["bp_idx"])
    n2, bp2, bss2, idx2 = run_second(f2, pk, both["info"], both["model"], bp1, scr, len(both["bp"]) + 64, len(both["bss"]) + 4096, lm_arrays=lma)
    assert n2 == len(both["bp"]) and np.array_equal(bp2, both["bp"]) and np.array_equal(bss2, both["bss"]) and np.array_equal(idx2, both["bp_idx"])
    # ps_seg_iter of the same decode from the tables alone (psb_result.cu): every segment's frames and scores
    from pocketsphinx_b200 import api
    full = refdrv.decode(hd, BIG_LM, dic, pcm, bestpath="no", compallsen="yes", pl_window="0", fwdflat="yes")
    entry, score, _ = api.ngram_hyp(bp2, idx2, both["n_frame"], both["finish_wid"])
    seg = api.ngram_segments(both["info"], both["model"], bp2, bss2, entry, lm_arrays=lma, second_pass=True)
    lines = [l.split() for l in full["seg"].split("\n") if l]
    assert score == full["score"] and len(lines) == len(seg) > 3
    for s, (word, sf, ef, ascr, lscr) in zip(seg, lines):
        assert (int(s[2]), int(s[3]), int(s[5]), int(s[6])) == (int(sf), int(ef), int(ascr), int(lscr)), word
