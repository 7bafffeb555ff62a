"""GPU: the GRU scan kernels of csrc/gru_scan.cu through the C-ABI (isa_gru_scan_fwd / isa_gru_scan_bwd) against the
float64 recurrence of oracle/gru_scan_ref.py, at every launch configuration the host can pick:

  * the tensor-core forward and backward (n_units = 100, 16-byte-aligned gx / stash, out, dout) at S = 4, 8, 12, 14
    and 16 sequences per CTA, the generic FFMA forward and backward at S = 4, 8 and 16, each with a partly filled last
    CTA and with more CTAs than SMs;
  * T from 1 (the backward's MMA issuer runs no step) past the depth of both TMA rings up to 512;
  * both real token maps of renet._geometry (rows, and columns with a nonzero outer stride);
  * one kernel family's forward feeding the other family's backward, b_ih passed or folded into gx, saturated gates,
    and W_hh at an address that is 4 but not 8 or 16-byte aligned.

Every output buffer is NaN-filled with a 16-byte guard on each side before a call: afterwards every element inside
must be written and the guards untouched.  test_cases_reach_every_launch_configuration mirrors the host's choice of S
and fails, naming the bucket, if the cases below stop reaching one of them."""
import collections
import math

import pytest
import torch

from oracle.gru_scan_ref import gru_scan_bwd, gru_scan_fwd

pytestmark = pytest.mark.gpu

RTOL = 2e-4                 # the ReNet tolerance of tests/test_renet_gpu.py
ISA_ERR_BAD_ARG = -1
GUARD = 4                   # floats: 16 bytes on each side of every buffer


# ---- mirrors of the host's launch choice (csrc/gru_scan.cu: pick_S_tc, pick_S, and the dispatch in isa_gru_scan_fwd /
# isa_gru_scan_bwd); keep them in step with the C++
def pick_S_tc(n_seq, num_sms):
    best, best_cost = 4, None
    for S in (16, 14, 12, 8, 4):
        waves = -(-2 * -(-n_seq // S) // num_sms)
        cost = waves * (6 + S)
        if best_cost is None or cost < best_cost:
            best, best_cost = S, cost
    return best


def pick_S(n_seq, num_sms):
    if -(-n_seq // 16) * 2 * 10 >= num_sms * 8:
        return 16
    if -(-n_seq // 8) * 2 * 10 >= num_sms * 8:
        return 8
    return 4


# gx_off / dout_off / whh_off: the operand starts one float past a 16-byte boundary.  An offset gx sends the forward to
# the generic kernel, an offset dout the backward; w_hh's alignment does not change the dispatch.
Case = collections.namedtuple("Case", "name B H W mode n b_ih gx_off dout_off whh_off sat")


def _c(name, B, H, W, mode, n, b_ih=True, gx_off=0, dout_off=0, whh_off=0, sat=False):
    return Case(name, B, H, W, mode, n, b_ih, gx_off, dout_off, whh_off, sat)


CASES = [
    # tensor cores (n = 100): one case per S bucket, each with a partly filled last CTA, T = 1 .. 6 spread over them
    _c("tc_one_seq_T1", 1, 1, 1, "hor", 100),
    _c("tc_S4_T2", 3, 5, 2, "hor", 100, b_ih=False),
    _c("tc_S8_T3", 3, 3, 101, "ver", 100),
    _c("tc_S12_T4", 7, 4, 101, "ver", 100, b_ih=False),
    _c("tc_S14_T5", 9, 111, 5, "hor", 100),
    _c("tc_S16_T6", 2, 6, 555, "ver", 100, b_ih=False),
    _c("tc_S16_T1", 1, 1, 1100, "ver", 100),
    _c("tc_two_waves_T7", 13, 100, 7, "hor", 100, b_ih=False),
    _c("tc_S8_dp_rank_T64", 8, 64, 64, "ver", 100),
    _c("tc_S4_T512", 1, 512, 256, "ver", 100),
    _c("tc_saturated", 4, 9, 250, "ver", 100, sat=True),
    _c("tc_w_hh_offset", 2, 8, 37, "ver", 100, whh_off=1),
    # one family's forward into the other family's backward; n = 100 on the generic kernels
    _c("tc_fwd_generic_bwd", 1, 700, 5, "hor", 100, dout_off=1),
    _c("generic_fwd_tc_bwd", 1, 1190, 3, "hor", 100, b_ih=False, gx_off=1),
    _c("generic_n100", 2, 9, 17, "ver", 100, gx_off=1, dout_off=1),
    # generic kernels
    _c("generic_n4", 2, 3, 7, "hor", 4, b_ih=False),
    _c("generic_n36_S8", 5, 9, 99, "ver", 36),
    _c("generic_n64_S16", 2, 5, 500, "ver", 64, b_ih=False),
    _c("generic_n128_S16_two_waves", 1, 1201, 3, "hor", 128),
    _c("generic_n128_S8_two_waves", 3, 3, 201, "ver", 128, b_ih=False),
    _c("generic_saturated", 2, 11, 13, "ver", 64, sat=True),
]


def _geom(c):
    from isa_b200.renet import _geometry
    return _geometry(c.B, c.H, c.W, c.mode)


def _launches(c, num_sms):
    """-> [(family, pass, S, n_seq, T, ctas)] of the forward and the backward of case c."""
    n_seq, T = _geom(c)[:2]
    res = []
    for pas, tc in (("fwd", c.n == 100 and not c.gx_off), ("bwd", c.n == 100 and not c.dout_off)):
        S = (pick_S_tc if tc else pick_S)(n_seq, num_sms)
        res.append(("tc" if tc else "generic", pas, S, n_seq, T, 2 * -(-n_seq // S)))
    return res


def _num_sms():
    import ctypes
    from isa_b200 import _lib
    v = ctypes.c_int(0)
    _lib.check(_lib.load().isa_num_sms(ctypes.byref(v)), "isa_num_sms")
    return v.value


def test_cases_reach_every_launch_configuration(cuda):
    num_sms = _num_sms()
    seen = [l for c in CASES for l in _launches(c, num_sms)]
    missing = []
    for fam, sizes in (("tc", (4, 8, 12, 14, 16)), ("generic", (4, 8, 16))):
        for pas in ("fwd", "bwd"):
            mine = [l for l in seen if l[0] == fam and l[1] == pas]
            for S in sizes:
                if not any(l[2] == S and l[3] % S for l in mine):
                    missing.append("%s %s S=%d with a partly filled last CTA" % (fam, pas, S))
            if not any(l[5] > num_sms for l in mine):
                missing.append("%s %s with more CTAs than the %d SMs" % (fam, pas, num_sms))
            if fam == "tc":
                for T in (1, 2, 3, 4, 5, 6):
                    if not any(l[4] == T for l in mine):
                        missing.append("tc %s T=%d" % (pas, T))
                if not any(l[4] > 64 for l in mine):
                    missing.append("tc %s T>64" % pas)
    assert not missing, "launch configurations no case reaches: %s" % "; ".join(missing)


def _guarded(numel, off, device, data=None):
    """(store, view): `numel` floats starting GUARD + off floats into a NaN-filled store, GUARD NaN floats after them."""
    store = torch.full((GUARD + off + numel + GUARD,), float("nan"), device=device)
    assert store.data_ptr() % 16 == 0
    view = store[GUARD + off:GUARD + off + numel]
    if data is not None:
        view.copy_(data.reshape(-1))
    return store, view


def _written(store, view, off, what):
    inside = store[GUARD + off:GUARD + off + view.numel()]
    assert not torch.isnan(inside).any(), "%s: %d elements not written" % (what, int(torch.isnan(inside).sum()))
    guards = torch.cat([store[:GUARD + off], store[GUARD + off + view.numel():]])
    assert torch.isnan(guards).all(), "%s: written outside the buffer" % what


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def _close(a, b, what):
    """max|a - b| / max|b| per direction (dim 1 of a [tokens][2][...] view)."""
    for d in range(2):
        e = _rel(a[:, d], b[:, d])
        assert e < RTOL, "%s, direction %d: relative error %.3e" % (what, d, e)


@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_gru_scan_against_float64(cuda, c):
    from isa_b200 import _lib
    lib = _lib.load()
    st = _lib.stream_ptr(cuda)
    n = c.n
    geom = _geom(c)
    tokens = c.B * c.H * c.W
    g = torch.Generator(device=cuda).manual_seed(CASES.index(c) + 1)
    k = 1.0 / math.sqrt(n)                      # nn.GRU's initialisation range

    def uni(*shape):
        return (torch.rand(*shape, generator=g, device=cuda) * 2 - 1) * k

    gx = torch.randn(tokens, 6 * n, generator=g, device=cuda) * (25.0 if c.sat else 1.0)
    w_hh = uni(2, 3 * n, n) * (4.0 if c.sat else 1.0)
    b_hh = uni(2, 3 * n)
    b_ih = uni(2, 3 * n) if c.b_ih else None
    dout = torch.randn(tokens, 2 * n, generator=g, device=cuda)
    _, gx_v = _guarded(gx.numel(), c.gx_off, cuda, gx)
    _, whh_v = _guarded(w_hh.numel(), c.whh_off, cuda, w_hh)
    _, dout_v = _guarded(dout.numel(), c.dout_off, cuda, dout)

    def fwd(with_stash=True):
        out_s, out = _guarded(tokens * 2 * n, 0, cuda)
        stash_s, stash = _guarded(tokens * 8 * n, 0, cuda) if with_stash else (None, None)
        _lib.check(lib.isa_gru_scan_fwd(_lib.ptr(gx_v), _lib.ptr(whh_v), _lib.ptr(b_hh), _lib.ptr(b_ih), geom[0], geom[1], n,
                                        *geom[2:], _lib.ptr(out), _lib.ptr(stash), st), "isa_gru_scan_fwd")
        torch.cuda.synchronize()
        _written(out_s, out, 0, "out")
        if with_stash:
            _written(stash_s, stash, 0, "stash")
        return out, stash

    def bwd(out, stash):
        dgx_s, dgx = _guarded(tokens * 6 * n, 0, cuda)
        dghn_s, dghn = _guarded(tokens * 2 * n, 0, cuda)
        _lib.check(lib.isa_gru_scan_bwd(_lib.ptr(dout_v), _lib.ptr(out), _lib.ptr(stash), _lib.ptr(whh_v), geom[0], geom[1], n,
                                        *geom[2:], _lib.ptr(dgx), _lib.ptr(dghn), st), "isa_gru_scan_bwd")
        torch.cuda.synchronize()
        _written(dgx_s, dgx, 0, "dgx")
        _written(dghn_s, dghn, 0, "dghn")
        return dgx, dghn

    out, stash = fwd()
    out_ref, stash_ref = gru_scan_fwd(gx_v.view(tokens, 6 * n), whh_v.view(2, 3 * n, n), b_hh, b_ih, *geom)
    _close(out.view(tokens, 2, n), out_ref.view(tokens, 2, n), "out")
    for qi, q in enumerate("r z n hn".split()):
        _close(stash.view(tokens, 2, 4, n)[:, :, qi], stash_ref.view(tokens, 2, 4, n)[:, :, qi], "stash " + q)

    dgx, dghn = bwd(out, stash)
    dgx_ref, dghn_ref = gru_scan_bwd(dout_v.view(tokens, 2 * n), gx_v.view(tokens, 6 * n), whh_v.view(2, 3 * n, n), b_hh, b_ih,
                                     *geom)
    _close(dgx.view(tokens, 2, 3 * n), dgx_ref, "dgx")
    _close(dghn.view(tokens, 2, n), dghn_ref, "dghn")

    # the stash is optional and changes nothing; the same call gives the same bits
    out_nostash, _ = fwd(with_stash=False)
    assert torch.equal(out_nostash, out), "out differs without a stash"
    out2, stash2 = fwd()
    assert torch.equal(out2, out) and torch.equal(stash2, stash), "forward is not deterministic"
    dgx2, dghn2 = bwd(out, stash)
    assert torch.equal(dgx2, dgx) and torch.equal(dghn2, dghn), "backward is not deterministic"


def test_gru_scan_rejects_bad_arguments(cuda):
    """Each bad argument returns ISA_ERR_BAD_ARG before anything runs: the NaN-filled outputs stay untouched."""
    from isa_b200 import _lib
    from isa_b200.renet import _geometry
    lib = _lib.load()
    st = _lib.stream_ptr(cuda)
    n, B, H, W = 8, 2, 3, 5
    tokens = B * H * W
    n_seq, T, inner, outer, inner_s, t_s = _geometry(B, H, W, "ver")
    gx = torch.randn(tokens, 6 * n, device=cuda)
    w_hh = torch.randn(2, 3 * n, n, device=cuda)
    b = torch.randn(2, 3 * n, device=cuda)
    dout = torch.randn(tokens, 2 * n, device=cuda)
    fwd_in = torch.randn(tokens, 2 * n, device=cuda)
    stash_in = torch.rand(tokens, 8 * n, device=cuda)
    outs = {name: torch.full((tokens, k * n), float("nan"), device=cuda)
            for name, k in (("out", 2), ("stash", 8), ("dgx", 6), ("dghn", 2))}
    P = _lib.ptr

    def fwd(**kw):
        a = dict(gx=P(gx), w_hh=P(w_hh), b_hh=P(b), b_ih=P(b), n_seq=n_seq, T=T, n=n, inner=inner,
                 out=P(outs["out"]), stash=P(outs["stash"]))
        a.update(kw)
        return lib.isa_gru_scan_fwd(a["gx"], a["w_hh"], a["b_hh"], a["b_ih"], a["n_seq"], a["T"], a["n"], a["inner"],
                                    outer, inner_s, t_s, a["out"], a["stash"], st)

    def bwd(**kw):
        a = dict(dout=P(dout), out=P(fwd_in), stash=P(stash_in), w_hh=P(w_hh), n_seq=n_seq, T=T, n=n, inner=inner,
                 dgx=P(outs["dgx"]), dghn=P(outs["dghn"]))
        a.update(kw)
        return lib.isa_gru_scan_bwd(a["dout"], a["out"], a["stash"], a["w_hh"], a["n_seq"], a["T"], a["n"], a["inner"],
                                    outer, inner_s, t_s, a["dgx"], a["dghn"], st)

    bad = [dict(n=0), dict(n=6), dict(n=132), dict(T=0), dict(n_seq=0), dict(inner=0)]
    calls = [("fwd", kw, fwd) for kw in bad + [dict(gx=None), dict(w_hh=None), dict(b_hh=None), dict(out=None)]]
    calls += [("bwd", kw, bwd) for kw in bad + [dict(dout=None), dict(out=None), dict(stash=None), dict(w_hh=None),
                                                 dict(dgx=None), dict(dghn=None)]]
    for pas, kw, fn in calls:
        rc = fn(**kw)
        assert rc == ISA_ERR_BAD_ARG, "%s %s: rc %d" % (pas, kw, rc)
        assert b"gru_scan" in lib.isa_last_error(), (pas, kw)
    torch.cuda.synchronize()
    for name, t in outs.items():
        assert torch.isnan(t).all(), "%s written by a rejected call" % name
