"""Host-buffer scoring entries (dist_b200_score_sample_batch_host, dist_b200_score_logp_batch_host) against the
device-pointer entries (score_sample_batch, score_logp_batch) on the same inputs: every result bit-identical, over each
route by which the host form stages rows:

  feature lists  nich and dpd sampling (row chunks alternate over the two streams), dpd logp, nich + dpd and niw at
                 d = 3 and d = 40 (one compute stream, the copies run ahead on the second), gp + bb (alternating, the
                 GammaPoisson value tables refreshed before the second stream starts)
  buffers        pageable (staged through the page-locked mirror), torch pin_memory and host_register (copied from
                 directly, or read in place by the zero-copy route), mixed (the first column page-locked, the other
                 columns and u pageable)
  chunking       DIST_B200_OPT_HOST_CHUNKS 1, 2, 3, 4 and 7 at N = 250 001, and N = 1000 (one chunk); page-locked
                 buffers under DIST_B200_OPT_HOST_ZEROCOPY 0 and 1
  outputs        assign, assign with the [N][G] scores, logp
"""
import contextlib

import numpy as np
import pytest

from distributions_b200 import capi, synth

pytestmark = pytest.mark.gpu

N_BIG = 250_001  # more than 7 x 32768 rows (the least chunk) and not a multiple of 256
WORKLOADS = {
    "nich": lambda n: [synth.nich(31, 70, n)],
    "dpd": lambda n: [synth.dpd(32, 50, n, V=100, other_frac=0.1)],
    "nich_dpd": lambda n: [synth.nich(33, 40, n), synth.dpd(34, 40, n, V=100, other_frac=0.1)],
    "niw3": lambda n: [synth.niw(35, 24, n, d=3)],
    "niw40": lambda n: [synth.niw(36, 24, n, d=40)],
    "gp_bb": lambda n: [synth.gp(37, 40, n), synth.bb(38, 40, n)],
}
ALL_OUTPUTS = ("assign", "assign_scores", "logp")
# feature list: (workload, outputs)
LISTS = {
    "nich": ("nich", ALL_OUTPUTS),
    "dpd_sample": ("dpd", ("assign", "assign_scores")),
    "dpd_logp": ("dpd", ("logp",)),
    "nich_dpd": ("nich_dpd", ALL_OUTPUTS),
    "niw3": ("niw3", ALL_OUTPUTS),
    "niw40": ("niw40", ALL_OUTPUTS),
    "gp_bb": ("gp_bb", ALL_OUTPUTS),
}
CASES = [(lst, out) for lst, (_, outs) in LISTS.items() for out in outs]
# (rows, DIST_B200_OPT_HOST_CHUNKS; 0 = the default)
CHUNKINGS = {"chunks1": (N_BIG, 1), "chunks2": (N_BIG, 2), "chunks3": (N_BIG, 3), "chunks4": (N_BIG, 4), "chunks7": (N_BIG, 7),
             "n1000": (1000, 0)}
# (buffers, DIST_B200_OPT_HOST_ZEROCOPY): the option only matters when every buffer is page-locked
BUFFER_RUNS = [("pageable", 0), ("pinned", 0), ("pinned", 1), ("registered", 0), ("registered", 1), ("mixed", 0)]
MODEL_ID = {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW, "bnb": capi.BNB}


@pytest.fixture(scope="module")
def ctx():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    _SETUPS.clear()
    c.close()


class Setup:
    """features, host columns, u and prior of one workload at n rows, and the device-pointer entries' results"""

    def __init__(self, ctx, workload, n):
        ws = WORKLOADS[workload](n)
        self.n = n
        self.feats = [ctx.feature(MODEL_ID[w["model"]]).update_all(w) for w in ws]
        self.cols = [np.ascontiguousarray(w["values"], dtype=capi.COLUMN_DTYPE[MODEL_ID[w["model"]]]) for w in ws]
        self.u = np.ascontiguousarray(ws[0]["u"], dtype=np.float32)
        self.prior = ctx.prior_pitman_yor_host(synth.PY_ALPHA, synth.PY_D, ws[0]["sizes"])
        self.ref = {}

    def device(self, ctx, out):
        import torch
        if out not in self.ref:
            n, G = self.n, self.feats[0].groups
            cols = [torch.from_numpy(c).cuda() for c in self.cols]
            prior = torch.from_numpy(self.prior).cuda()
            if out == "logp":
                res = [torch.full((n,), 777.0, device="cuda", dtype=torch.float32)]
                ctx.score_logp_batch(self.feats, cols, n, prior, res[0])
            else:
                res = [torch.full((n,), -5, device="cuda", dtype=torch.int32)]
                if out == "assign_scores":
                    res.append(torch.full((n, G), 777.0, device="cuda", dtype=torch.float32))
                ctx.score_sample_batch(self.feats, cols, n, prior, torch.from_numpy(self.u).cuda(), res[0], res[1] if len(res) > 1 else None)
            torch.cuda.synchronize()
            self.ref[out] = [t.cpu().numpy() for t in res]
        return self.ref[out]


_SETUPS = {}


def setup(ctx, lst, n):
    key = (LISTS[lst][0], n)
    if key not in _SETUPS:
        _SETUPS[key] = Setup(ctx, key[0], n)
    return _SETUPS[key]


@contextlib.contextmanager
def buffers(ctx, s, out, kind):
    """(columns, u, output array) of one buffer kind; the output starts as a sentinel"""
    import torch
    dtype = np.float32 if out == "logp" else np.int32
    fresh = lambda: np.full(s.n, -7, dtype)  # noqa: E731
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()  # noqa: E731
    if kind == "pageable":
        yield s.cols, s.u, fresh()
    elif kind == "pinned":
        yield [pin(c) for c in s.cols], pin(s.u), pin(fresh())
    elif kind == "mixed":
        yield [pin(s.cols[0])] + s.cols[1:], s.u, fresh()
    else:
        reg = [c.copy() for c in s.cols] + [s.u.copy(), fresh()]
        for a in reg:
            ctx.host_register(a)
        try:
            yield reg[:-2], reg[-2], reg[-1]
        finally:
            for a in reg:
                ctx.host_unregister(a)


def call_host(ctx, s, out, cols, u, dst):
    if out == "logp":
        return [ctx.score_logp_batch_host(s.feats, cols, s.prior, logp_out=dst).copy()]
    assign, scores = ctx.score_sample_batch_host(s.feats, cols, s.prior, u, want_scores=out == "assign_scores", assign_out=dst)
    return [assign.copy()] + ([] if scores is None else [scores])


def run_host(ctx, s, out, kind, chunks, zerocopy):
    """the host entry's results for one configuration; the options are restored before it returns"""
    with buffers(ctx, s, out, kind) as (cols, u, dst):
        ctx.set_option(capi.OPT_HOST_CHUNKS, chunks)
        ctx.set_option(capi.OPT_HOST_ZEROCOPY, zerocopy)
        try:
            return call_host(ctx, s, out, cols, u, dst)
        finally:
            ctx.set_option(capi.OPT_HOST_CHUNKS, 0)
            ctx.set_option(capi.OPT_HOST_ZEROCOPY, 0)


@pytest.mark.parametrize("chunking", CHUNKINGS)
@pytest.mark.parametrize("lst,out", CASES)
def test_host_entry_matches_device(ctx, lst, out, chunking):
    n, chunks = CHUNKINGS[chunking]
    s = setup(ctx, lst, n)
    want = s.device(ctx, out)
    for kind, zerocopy in BUFFER_RUNS:
        got = run_host(ctx, s, out, kind, chunks, zerocopy)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert np.array_equal(g, w), "%s %s %s: buffers %s, zero-copy option %d" % (lst, out, chunking, kind, zerocopy)
