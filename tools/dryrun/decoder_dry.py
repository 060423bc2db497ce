# Dry run of pocketsphinx_b200.decoder.Decoder on the CPU: the device stages are replaced by the compiled reference
# (front end, scorer, phone loop: oracle/_ref) and by the host emulation of the search kernels (conftest_dry.FakeCtx);
# the Decoder's own code -- file loading, argument plumbing, table sizes, hypothesis and segment extraction -- runs
# unchanged and must reproduce a plain reference decode (words, score, every segment).  Run by tools/dryrun/run.sh.
import os, sys, types
import numpy as np
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE))); sys.path.insert(0, HERE)
import conftest_dry as D
from oracle import refdrv
from pocketsphinx_b200 import api as real_api, decoder

REF = os.path.dirname(refdrv.LIB_PATH)
HD, DIC, LM = os.path.join(REF, "model", "en-us"), os.path.join(REF, "data", "turtle.dic"), os.path.join(REF, "data", "turtle.lm.bin")


class FE:
    sample_offsets = staticmethod(real_api.FrontEnd.sample_offsets)
    def __init__(self, desc, device=0): self.desc = desc
    def close(self): pass

class Model:
    def __init__(self, pm, device=0): self.pm = pm
    def close(self): pass

class PhoneLoop:
    def __init__(self, ctx, ssid, tmatid, window, beam, pbeam, pip, weight):
        assert (window, beam, pbeam, pip, weight) == (5, -225, -225, 0, 3.0) and len(ssid) == len(tmatid) == 42
        self.n_phones = len(ssid)
    def close(self): pass

class Batch:
    def __init__(self, model, max_utts, max_frames): self.model = model
    def decode_pcm_host(self, fe, pl, pcm, off):
        scr, pen, foff = [], [], [0]
        for u in range(len(off) - 1):
            x = pcm[off[u]:off[u + 1]]
            ref = refdrv.RefModel(HD); scr.append(np.ascontiguousarray(ref.score(ref.featurize_fresh(x)))); ref.close()
            ref = refdrv.RefModel(HD); pen.append(np.ascontiguousarray(ref.phoneloop(x)["pen"], np.int32)); ref.close()
            foff.append(foff[-1] + len(scr[-1]))
        self.scr = np.ascontiguousarray(np.concatenate(scr))
        return np.array(foff, np.int32), None, np.concatenate(pen)
    def senscr_device_ptr(self): return self.scr.ctypes.data
    def close(self): pass

decoder.api = types.SimpleNamespace(FrontEnd=FE, Model=Model, Batch=Batch, PhoneLoop=PhoneLoop, HmmContext=D.FakeCtx,
                                    ngram_hyp=real_api.ngram_hyp, ngram_segments=real_api.ngram_segments, PsbError=real_api.PsbError)
go = np.fromfile(os.path.join(REF, "data", "goforward.raw"), np.int16)
utts = [go, go[:30000]]
dec = decoder.Decoder(HD, DIC, LM)
out = dec.decode_raw_batch(utts)
dec.close()
for pcm, o in zip(utts, out):
    # the device scores every senone of every frame, i.e. the reference with -compallsen yes (per-frame normalisation
    # by the best of ALL senones; with the default active-list evaluation path scores shift, words do not)
    want = refdrv.decode(HD, LM, DIC, pcm, bestpath="no", compallsen="yes")
    assert refdrv.decode(HD, LM, DIC, pcm, bestpath="no")["hyp"] == want["hyp"]
    lines = [l.split() for l in want["seg"].split("\n") if l]
    assert o["hyp"] == want["hyp"] and o["score"] == want["score"], (o["hyp"], want["hyp"], o["score"], want["score"])
    assert len(lines) == len(o["seg"])
    for s, w, (word, sf, ef, ascr, lscr) in zip(o["seg"], o["words"], lines):
        assert (w, int(s[2]), int(s[3]), int(s[5]), int(s[6])) == (word, int(sf), int(ef), int(ascr), int(lscr)), (w, s, word)
    print("decoder dry run:", repr(o["hyp"]), o["score"], len(o["seg"]), "segments == reference")
