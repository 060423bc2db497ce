"""CPU, build container (needs oracle/_ref/libpsref.so and the turtle LM next to the reference
sources): the reference's first pass run LIVE on shuffled, rescaled, noisy variants of goforward.raw
and under random beams / pruning limits / penalties / look-ahead windows, against (1) the oracle
restatement and (2) the host build of the device first pass's phase code in both thread orders.
Every backpointer-table row, the score stack and bp_table_idx must agree.
PSB_NGS_FUZZ_SEEDS=a:b widens the range (45 seeds were run when this was written: 0 mismatches)."""
import os
import random

import numpy as np
import pytest

from oracle import oracle, refdrv
from test_ngf_emul import emuls, run_second  # noqa: F401  (fixture)
from test_ngs_emul import emul, run_emul  # noqa: F401  (fixture)

pytestmark = pytest.mark.skipif(not refdrv.available(), reason="oracle/_ref/libpsref.so not built")
REF = os.path.dirname(refdrv.LIB_PATH)
LM, DIC = os.path.join(REF, "data", "turtle.lm.bin"), os.path.join(REF, "data", "turtle.dic")
needs_lm = pytest.mark.skipif(not os.path.exists(LM), reason="oracle/_ref/data/turtle.lm.bin not built")
HD = os.path.join(REF, "model", "en-us")


def _seeds():
    a, b = (int(x) for x in os.environ.get("PSB_NGS_FUZZ_SEEDS", "0:4").split(":"))
    return list(range(a, b))


def _score(pcm):
    ref = refdrv.RefModel(HD)
    pk = ref.packed()
    scr = np.ascontiguousarray(ref.score(ref.featurize_fresh(pcm)))
    ref.close()
    return pk, scr


def _check(emul, pk, scr, r, **la):
    got = oracle.fwdtree_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:r["n_ci"]], r["info"], r["model"], scr, **la)
    assert np.array_equal(got[0], r["bp"]) and np.array_equal(got[1], r["bss"]) and np.array_equal(got[2], r["bp_idx"])
    n, bp, bss, idx = run_emul(emul, pk, r["info"], r["model"], scr, len(r["bp"]) + 8, len(r["bss"]) + 64, **la)
    assert n == len(r["bp"]) and np.array_equal(bp, r["bp"])
    assert np.array_equal(bss, r["bss"]) and np.array_equal(idx, r["bp_idx"])


@needs_lm
@pytest.mark.parametrize("seed", _seeds())
def test_other_audio(emul, seed):  # noqa: F811
    go = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
    rng = np.random.default_rng(seed)
    pieces = np.split(go, np.sort(rng.integers(0, len(go), 6)))
    pcm = np.concatenate([pieces[i] for i in rng.permutation(len(pieces))]).astype(np.float64)
    pcm = pcm * rng.uniform(0.3, 1.5) + rng.normal(0, rng.uniform(0, 1500), len(pcm))
    pcm = np.clip(pcm, -32768, 32767).astype(np.int16)
    kv = [{}, dict(beam="1e-70", pbeam="1e-60", wbeam="1e-40", lpbeam="1e-50", lponlybeam="1e-40"),
          dict(maxwpf="6", maxhmmpf="400")][seed % 3]
    pk, scr = _score(pcm)
    _check(emul, pk, scr, refdrv.fwdtree(HD, LM, DIC, pcm, **kv))


@needs_lm
@pytest.mark.parametrize("seed", _seeds())
def test_other_settings(emul, seed):  # noqa: F811
    pcm = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
    rng = random.Random(seed)
    e = lambda a, b: "1e-%d" % rng.randint(a, b)  # noqa: E731
    kv = {}
    if rng.random() < 0.7:
        kv.update(beam=e(20, 90), pbeam=e(15, 90), wbeam=e(5, 60), lpbeam=e(10, 70), lponlybeam=e(5, 60))
    if rng.random() < 0.4:
        kv["maxwpf"] = str(rng.randint(1, 30))
    if rng.random() < 0.4:
        kv["maxhmmpf"] = str(rng.randint(20, 3000))
    if rng.random() < 0.4:
        kv.update(lw="%.1f" % rng.uniform(1, 12), wip="%.2f" % rng.uniform(0.1, 1), pip="%.2f" % rng.uniform(0.3, 1),
                  nwpen="%.2f" % rng.uniform(0.3, 1))
    la = {}
    if rng.random() < 0.5:
        kv["pl_window"] = str(rng.randint(1, 10))
        if rng.random() < 0.5:
            kv["pl_weight"] = "%.1f" % rng.uniform(0.5, 6)
        ref = refdrv.RefModel(HD)
        pl = ref.phoneloop(pcm, **{k: v for k, v in kv.items() if k.startswith("pl_")})
        ref.close()
        la = dict(pl_pen=pl["pen"], pl_window=int(kv["pl_window"]))
    pk, scr = _score(pcm)
    _check(emul, pk, scr, refdrv.fwdtree(HD, LM, DIC, pcm, **kv), **la)


@needs_lm
@pytest.mark.parametrize("seed", _seeds())
def test_both_passes_other_audio_and_settings(emuls, seed):  # noqa: F811
    """Second pass (ngram_search_fwdflat.c) chained behind the first, both through the phase code."""
    f1, f2 = emuls
    go = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
    rng = np.random.default_rng(1000 + seed)
    pieces = np.split(go, np.sort(rng.integers(0, len(go), 4)))
    pcm = np.concatenate([pieces[i] for i in rng.permutation(len(pieces))]).astype(np.float64)
    pcm = np.clip(pcm * rng.uniform(0.5, 1.2) + rng.normal(0, rng.uniform(0, 800), len(pcm)), -32768, 32767).astype(np.int16)
    kv = [dict(), dict(fwdflatbeam="1e-70", fwdflatwbeam="1e-30", fwdflatefwid="2", fwdflatsfwin="40"),
          dict(fwdflatbeam="1e-40", fwdflatwbeam="1e-12", fwdflatlw="11", maxwpf="10"),
          dict(fwdflatefwid="6", fwdflatsfwin="8", lw="4", fwdflatlw="9.5", pip="0.8")][seed % 4]
    pk, scr = _score(pcm)
    r = refdrv.fwdtree(HD, LM, DIC, pcm, fwdflat="yes", **kv)
    nc = r["n_ci"]
    n1, bp1, _, _ = run_emul(f1, pk, r["info"], r["model"], scr, 16384, 1 << 19)
    assert n1 >= 0
    want1 = oracle.fwdtree_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], r["info"], r["model"], scr)[0]
    assert np.array_equal(bp1, want1)
    got = oracle.fwdflat_run(pk["tp"], pk["sseq"], pk["phone_tmat"][:nc], pk["phone_ssid"][:nc], r["info"], r["model"], bp1, scr)
    assert np.array_equal(got[0], r["bp"]) and np.array_equal(got[1], r["bss"]) and np.array_equal(got[2], r["bp_idx"])
    n, bp, bss, idx = run_second(f2, pk, r["info"], r["model"], bp1, scr, len(r["bp"]) + 8, len(r["bss"]) + 64)
    assert n == len(r["bp"]) and np.array_equal(bp, r["bp"])
    assert np.array_equal(bss, r["bss"]) and np.array_equal(idx, r["bp_idx"])
