# Dry run of the gated GPU tests on the CPU: torch's .cuda() becomes the identity and HmmContext's search
# methods are served by the host emulation harnesses (same argument conventions as the real API).
# PSB_ROOT: the repository (run.sh copies this file out of it); PSB_EMUL_DIR: where lib{fsg,ngs,ngf}emul.so were built.
import ctypes as C, os, sys
import numpy as np
import pytest
ROOT = os.environ.get("PSB_ROOT") or os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
exec(open(os.path.join(ROOT, "tests", "conftest.py")).read().replace("os.path.dirname(os.path.dirname(os.path.abspath(__file__)))", repr(ROOT)))
import torch
torch.Tensor.cuda = lambda self, *a, **k: self
_to = torch.Tensor.to
torch.Tensor.to = lambda self, *a, **k: self if (a and isinstance(a[0], torch.device) and a[0].type == "cuda") else _to(self, *a, **k)
import test_fsg_emul as TF, test_ngs_emul as TN, test_ngf_emul as TG

class FakeCtx:
    def __init__(self, tp, sseq, n_sen, device=0):
        self.m = dict(tp=tp, sseq=sseq, phone_tmat=None, phone_ssid=None); self.n_sen = n_sen
        self.L = {k: C.CDLL(os.path.join(os.environ["PSB_EMUL_DIR"], "lib%semul.so" % k)) for k in ("fsg", "ngs", "ngf")}
        self.f_fsg = self.L["fsg"].fsg_emul_run; self.f_fsg.restype = C.c_int32; self.f_fsg.argtypes = TF.ARGT
        self.f1 = self.L["ngs"].ngs_emul_run; self.f1.restype = C.c_int32; self.f1.argtypes = TN.ARGT
        self.f2 = self.L["ngf"].ngf_emul_run; self.f2.restype = C.c_int32; self.f2.argtypes = TG.ARGT
    def _scr(self, ptr, utt_off, u):
        T = int(utt_off[u + 1] - utt_off[u])
        a = (C.c_int16 * (T * self.n_sen)).from_address(ptr + int(utt_off[u]) * self.n_sen * 2)
        return np.frombuffer(a, np.int16).reshape(T, self.n_sen).copy()
    def _pen(self, ptr, utt_off, u, n_ci):
        if not ptr: return None
        T = int(utt_off[u + 1] - utt_off[u])
        a = (C.c_int32 * (T * n_ci)).from_address(ptr + int(utt_off[u]) * n_ci * 4)
        return np.frombuffer(a, np.int32).reshape(T, n_ci).copy()
    def fsg(self, ptr, utt_off, g, cap):
        hs, ns = [], []
        for u in range(len(utt_off) - 1):
            h, n = TF._run(self.f_fsg, self.m, g, self._scr(ptr, utt_off, u), max(cap, 20000))
            hs.append(h[:cap]); ns.append(n)
        return hs, np.array(ns, np.int32)
    def ngram_fwdtree(self, ptr, utt_off, info, model, cit, bp_cap, bss_cap, d_pen_ptr=None, pl_window=0, lm_arrays=None):
        m = dict(self.m, phone_tmat=np.asarray(cit)); out = []
        for u in range(len(utt_off) - 1):
            pen = self._pen(d_pen_ptr, utt_off, u, len(cit))
            n, bp, bss, idx = TN.run_emul(self.f1, m, info, model, self._scr(ptr, utt_off, u), bp_cap, bss_cap, pl_pen=pen, pl_window=pl_window, lm_arrays=lm_arrays)
            if n < 0:
                from pocketsphinx_b200._lib import PsbError
                raise PsbError("overflow")
            out.append((bp, bss, idx))
        return out
    def ngram_fwdflat(self, ptr, utt_off, info, model, cit, cis, firsts, bp_cap, bss_cap, lm_arrays=None):
        m = dict(self.m, phone_tmat=np.asarray(cit), phone_ssid=np.asarray(cis)); out = []
        for u in range(len(utt_off) - 1):
            n, bp, bss, idx = TG.run_second(self.f2, m, info, model, firsts[u], self._scr(ptr, utt_off, u), bp_cap, bss_cap, lm_arrays=lm_arrays)
            if n < 0:
                from pocketsphinx_b200._lib import PsbError
                raise PsbError("overflow")
            out.append((bp, bss, idx))
        return out
    def ngram_two_pass(self, ptr, utt_off, info, model, cit, cis, bp_cap, bss_cap, d_pen_ptr=None, pl_window=0, first_cap=None, first_bss_cap=None, lm_arrays=None):
        first = self.ngram_fwdtree(ptr, utt_off, info, model, cit, first_cap or bp_cap, first_bss_cap or bss_cap, d_pen_ptr, pl_window, lm_arrays)
        return self.ngram_fwdflat(ptr, utt_off, info, model, cit, cis, [f[0] for f in first], bp_cap, bss_cap, lm_arrays), np.array([len(f[0]) for f in first], np.int32)
    def close(self): pass

class FakeApi:
    HmmContext = FakeCtx
    @staticmethod
    def device_count(): return 1

@pytest.fixture(scope="module")
def api():
    return FakeApi
