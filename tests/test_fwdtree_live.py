"""CPU, build container (needs oracle/_ref/libpsref.so): the first-pass restatement
(pso_fwdtree_run) against the reference's own ngram_search_fwdtree run LIVE in settings no fixture
holds -- other look-ahead windows / weights (penalties from the reference's phone loop), language
weights, pruning limits -- entry for entry on the backpointer table and the right-context stack."""
import os

import numpy as np
import pytest

from oracle import oracle, refdrv
from test_ngf_emul import emuls, run_second  # noqa: F401  (fixture)

pytestmark = pytest.mark.skipif(not refdrv.available(), reason="oracle/_ref/libpsref.so not built")
REF = os.path.dirname(refdrv.LIB_PATH)
LM, DIC = os.path.join(REF, "data", "turtle.lm.bin"), os.path.join(REF, "data", "turtle.dic")
needs_lm = pytest.mark.skipif(not os.path.exists(LM), reason="oracle/_ref/data/turtle.lm.bin not built")


@pytest.fixture(scope="module")
def scored():
    ref = refdrv.RefModel(os.path.join(REF, "model", "en-us"))
    pcm = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
    pk = ref.packed()
    scr = np.ascontiguousarray(ref.score(ref.featurize_fresh(pcm)))
    ref.close()
    return pk, pcm, scr


@needs_lm
@pytest.mark.parametrize("kv", [
    dict(pl_window="2", pl_beam="1e-5", pl_pbeam="1e-3"),
    dict(pl_window="9", pl_weight="1.5", beam="1e-40"),
    dict(pl_window="1", pl_weight="6", pl_pip="0.5", maxwpf="8"),
    dict(lw="3", wip="0.9", maxhmmpf="200"),
    dict(lw="12", beam="1e-60", wbeam="1e-40", lpbeam="1e-50", lponlybeam="1e-40", maxwpf="3"),
])
def test_fwdtree_settings_match_reference(scored, kv):
    pk, pcm, scr = scored
    hd = os.path.join(REF, "model", "en-us")
    r = refdrv.fwdtree(hd, LM, DIC, pcm, **kv)
    la = {}
    if "pl_window" in kv:
        ref = refdrv.RefModel(hd)                                # a fresh phone loop: its settings stick to the object
        pl = ref.phoneloop(pcm, **{k: v for k, v in kv.items() if k.startswith("pl_")})
        ref.close()
        assert pl["params"]["window"] == int(kv["pl_window"])
        la = dict(pl_pen=pl["pen"], pl_window=int(kv["pl_window"]))
    bp, bss, bp_idx = oracle.fwdtree_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:r["n_ci"]], r["info"], r["model"], scr, **la)
    assert bp.shape == r["bp"].shape and np.array_equal(bp, r["bp"])
    assert np.array_equal(bss, r["bss"]) and np.array_equal(bp_idx, r["bp_idx"])
    b, score = oracle.fwdtree_find_exit(bp, bp_idx, r["n_frame"], r["finish_wid"])
    assert score == r["score"]
    assert oracle.fwdtree_hyp(bp, b, r["words"], r["vocab"], r["start_wid"], r["finish_wid"]) == r["hyp"]


@needs_lm
@pytest.mark.parametrize("kv", [
    dict(fwdflatefwid="1", fwdflatsfwin="60", fwdflatlw="12"),
    dict(fwdflatlw="3.3", lw="7.1", pip="0.6", beam="1e-30"),
    dict(maxwpf="4", maxhmmpf="100", pl_window="3"),
])
def test_both_passes_match_reference(scored, kv):
    """First pass (with look-ahead where asked) chained into the second (ngram_search_fwdflat.c)."""
    pk, pcm, scr = scored
    hd = os.path.join(REF, "model", "en-us")
    r = refdrv.fwdtree(hd, LM, DIC, pcm, fwdflat="yes", **kv)
    nc = r["n_ci"]
    la = {}
    if "pl_window" in kv:
        ref = refdrv.RefModel(hd)
        pl = ref.phoneloop(pcm, **{k: v for k, v in kv.items() if k.startswith("pl_")})
        ref.close()
        la = dict(pl_pen=pl["pen"], pl_window=int(kv["pl_window"]))
    bp1, _, _ = oracle.fwdtree_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], r["info"], r["model"], scr, **la)
    bp, bss, bp_idx = oracle.fwdflat_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], pk["phone_ssid"][:nc], r["info"],
                                         r["model"], bp1, scr)
    assert bp.shape == r["bp"].shape and np.array_equal(bp, r["bp"])
    assert np.array_equal(bss, r["bss"]) and np.array_equal(bp_idx, r["bp_idx"])
    b, score = oracle.fwdtree_find_exit(bp, bp_idx, r["n_frame"], r["finish_wid"])
    assert score == r["score"]
    assert oracle.fwdtree_hyp(bp, b, r["words"], r["vocab"], r["start_wid"], r["finish_wid"]) == r["hyp"]


@needs_lm
@pytest.mark.parametrize("kv", [dict(), dict(fwdflatbeam="1e-40", fwdflatwbeam="1e-15", fwdflatlw="5")])
def test_second_pass_alone_matches_reference(emuls, scored, kv):  # noqa: F811
    """-fwdtree no -fwdflat yes: the flat search over the whole LM vocabulary, frame-synchronous
    (oracle restatement and the device second pass's phase code without a first-pass table)."""
    pk, pcm, scr = scored
    hd = os.path.join(REF, "model", "en-us")
    r = refdrv.fwdtree(hd, LM, DIC, pcm, fwdtree="no", fwdflat="yes", **kv)
    nc = r["n_ci"]
    bp, bss, bp_idx = oracle.fwdflat_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], pk["phone_ssid"][:nc], r["info"], r["model"],
                                         None, scr)
    assert bp.shape == r["bp"].shape and np.array_equal(bp, r["bp"])
    assert np.array_equal(bss, r["bss"]) and np.array_equal(bp_idx, r["bp_idx"])
    n, bp, bss, bp_idx = run_second(emuls[1], pk, r["info"], r["model"], None, scr, len(r["bp"]) + 8, len(r["bss"]) + 64)
    assert n == len(r["bp"]) and np.array_equal(bp, r["bp"]) and np.array_equal(bss, r["bss"]) and np.array_equal(bp_idx, r["bp_idx"])
