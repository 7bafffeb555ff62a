"""GPU: the discriminative-loss kernels of csrc/disc_loss.cu through the C-ABI (isa_disc_loss_fwd / isa_disc_loss_bwd)
against the float64 restatement oracle/disc_loss_torch.py run on the same device, on every route the host can pick:

  * the label-map kernel with per-warp accumulators (priv = 1) at every padded channel count CP = 8, 16, 24, 32, 64,
    with several CTAs per image and with one, and with one CTA accumulator (priv = 0: K (C + 1) too large);
  * the column walk on a label map (bs above the label-map kernel's co-resident CTAs, so it loops over images), on the
    label map distilled from a dense one-hot target, and on soft / overlapping dense masks (f32, i64, u8);
  * the column walk's early exit followed by the label-map kernel for one-hot dense targets.
isa_disc_loss_plan reports the route of every case; test_cases_reach_every_route fails, naming the route, if the cases
stop reaching one.  Semantics: all four terms, norm 1 and 2, normalize_means on and off, q_den, grad_loss, grad_means,
n_objects of 0, below 0 and above K, all-background images, labels in [K, 255), tiny and one-pixel-wide images.

Every output buffer sits between 16-byte guards in a store filled with a NaN bit pattern no arithmetic produces:
afterwards every element inside must be written and the guards untouched.  The forward runs on a workspace filled with
0xFF bytes and again on a zeroed one: the label-map kernel with priv = 1 must give the same bits, the routes with float
atomics the same values within tolerance."""
import collections
import ctypes

import numpy as np
import pytest
import torch

from isa_b200 import synth
from oracle import disc_loss_torch as R

pytestmark = pytest.mark.gpu

ISA_ERR_BAD_ARG, ISA_ERR_UNSUPPORTED, ISA_ERR_WORKSPACE = -1, -2, -3
ROUTE_LAB, ROUTE_COL_THEN_LAB, ROUTE_COL = 0, 1, 2
ROUTE_NAMES = {ROUTE_LAB: "lab", ROUTE_COL_THEN_LAB: "col+lab", ROUTE_COL: "col"}
KINDS = {"label": 0, "f32": 1, "i64": 2, "u8": 3}
DTYPES = {"f32": np.float32, "i64": np.int64, "u8": np.uint8}
GUARD = 4                       # 32-bit words: 16 bytes on each side of every buffer
SENTINEL = 0x7FC0DEAD           # a quiet NaN with a payload no kernel arithmetic produces
DV, DD = 0.5, 1.5
SHIPPED = (1.0, 0.0, 0.0, 0.005)
ALL_TERMS = (1.0, 1.0, 0.001, 0.005)
RTOL = 1e-4                     # loss and terms, relative (tests/test_disc_loss_gpu.py)
MEANS_ATOL = 1e-5
GRAD_RTOL = 1e-4                # of the gradient's largest element

# tgt: onehot | soft (f32 weights, overlapping) | overlap (integer masks with second entries and values of 2)
#      | single_w (one-hot but one pixel with weight != 1) | high_ch (overlapping entries only in channels >= n_objects)
# nobj: None = the synthetic counts, else a list; bg: "image" (image 0 all background) or "batch"; hi: labels in [K, 255)
# q: None, "local" (q_den = the local foreground count: same bits as NULL) or "x1.7"; gm: "rand", "zeros" (vs NULL) or None
Case = collections.namedtuple("Case", "name kind bs C K H W tgt norm normalize terms q gl gm nobj bg hi n_max")


def _c(name, kind, bs, C, K, H, W, tgt="onehot", norm=2, normalize=True, terms=SHIPPED, q=None, gl=1.0, gm="rand", nobj=None,
       bg=None, hi=False, n_max=None):
    return Case(name, kind, bs, C, K, H, W, tgt, norm, normalize, terms, q, gl, gm, nobj, bg, hi, n_max)


CASES = [
    # label-map kernel, priv = 1, several CTAs per image, one case per CP bucket (C = 1, 8 | 9 | 17, 24 | 25, 32 | 33, 64)
    _c("lab_C1", "label", 2, 1, 3, 40, 50),
    _c("lab_C8", "label", 3, 8, 8, 37, 45),
    _c("lab_C9", "label", 2, 9, 5, 33, 70),
    _c("lab_C17", "label", 2, 17, 12, 50, 41, q="local"),
    _c("lab_C24", "label", 2, 24, 32, 64, 64),
    _c("lab_C25", "label", 2, 25, 20, 45, 45),
    _c("lab_C32", "label", 2, 32, 40, 48, 48, n_max=40),
    _c("lab_C33", "label", 2, 33, 10, 40, 40),
    _c("lab_C64", "label", 2, 64, 16, 40, 40, gm="zeros"),
    # ... one CTA per image: images of at most 256 pixels, or more images than co-resident CTAs / 2
    _c("lab_C1_H1", "label", 3, 1, 2, 1, 200),
    _c("lab_C8_7x9", "label", 2, 8, 4, 7, 9),
    _c("lab_C9_W1", "label", 2, 9, 3, 50, 1),
    _c("lab_C17_15x17", "label", 2, 17, 5, 15, 17),
    _c("lab_C24_bs200", "label", 200, 24, 8, 16, 16),
    _c("lab_C25_3x31", "label", 2, 25, 4, 3, 31),
    _c("lab_C32_11x13", "label", 2, 32, 6, 11, 13),
    _c("lab_C33_H1", "label", 2, 33, 4, 1, 33),
    _c("lab_C64_9x9", "label", 2, 64, 5, 9, 9),
    # label-map kernel, priv = 0
    _c("lab_priv0_C64_K64", "label", 2, 64, 64, 40, 40, n_max=64, terms=ALL_TERMS),
    _c("lab_priv0_C24_K254", "label", 2, 24, 254, 48, 48, n_max=120),
    # column walk on a label map, looping over images (bs above the co-resident CTAs, and above 640)
    _c("col_label_bs700", "label", 700, 24, 8, 3, 5),
    _c("col_label_C8_bs300", "label", 300, 8, 4, 8, 40, terms=ALL_TERMS, norm=1),
    # column walk on the label map distilled from a dense one-hot target
    _c("col_onehot_f32", "f32", 300, 12, 6, 6, 10),
    _c("col_onehot_i64", "i64", 300, 12, 6, 6, 10, terms=ALL_TERMS),
    _c("col_onehot_u8", "u8", 300, 12, 6, 6, 10, norm=1),
    # column walk exits at once, then the label-map kernel (compared bit for bit with the label map below)
    _c("onehot_f32", "f32", 3, 16, 8, 30, 40),
    _c("onehot_i64", "i64", 3, 16, 8, 30, 40, terms=ALL_TERMS),
    _c("onehot_u8", "u8", 3, 16, 8, 30, 40, norm=1),
    # column walk on dense masks that are not one-hot (read_mask_k and the dense backward)
    _c("soft_f32", "f32", 2, 12, 5, 20, 24, tgt="soft"),
    _c("overlap_i64", "i64", 2, 10, 6, 24, 30, tgt="overlap"),
    _c("overlap_u8", "u8", 3, 20, 7, 26, 26, tgt="overlap", terms=ALL_TERMS),
    _c("soft_f32_bs300", "f32", 300, 8, 3, 4, 6, tgt="soft"),
    _c("overlap_C64", "f32", 2, 64, 4, 12, 12, tgt="soft", terms=ALL_TERMS),
    _c("single_w_f32", "f32", 2, 8, 4, 16, 16, tgt="single_w"),
    _c("single_w_i64", "i64", 2, 8, 4, 16, 16, tgt="single_w", q="local"),
    _c("high_ch_f32", "f32", 2, 8, 6, 16, 20, tgt="high_ch", nobj=[2, 3]),
    _c("high_ch_u8", "u8", 2, 8, 6, 16, 20, tgt="high_ch", nobj=[3, 2]),
    # the column walk at the largest K whose shared memory fits at C = 64 (on a B200)
    _c("soft_C64_K213", "f32", 2, 64, 213, 8, 8, tgt="soft"),
    # n_objects of 0, below 0 and above K; all-background images; labels in [K, 255)
    _c("nobj_edges_lab", "label", 3, 8, 5, 24, 24, nobj=[0, -2, 9], n_max=5),
    _c("nobj_edges_col", "f32", 3, 8, 5, 24, 24, tgt="soft", nobj=[0, -2, 9]),
    _c("bg_image_lab", "label", 2, 8, 4, 20, 20, bg="image"),
    _c("bg_image_col", "u8", 2, 8, 4, 20, 20, tgt="overlap", bg="image"),
    _c("bg_batch_lab", "label", 2, 8, 4, 20, 20, bg="batch"),
    _c("bg_batch_i64", "i64", 2, 8, 4, 20, 20, bg="batch"),
    _c("hi_labels_lab", "label", 2, 8, 4, 20, 20, hi=True, terms=ALL_TERMS),
    _c("hi_labels_col", "label", 300, 8, 4, 6, 6, hi=True),
    _c("absent_instance_lab", "label", 2, 8, 6, 20, 20, nobj=[4, 7], n_max=3),
]
# every term, both norms, means normalised or not, at both forward kernels; q_den, grad_loss and grad_means
for _kern, _kind, _tgt in (("lab", "label", "onehot"), ("col", "f32", "soft")):
    for _norm in (1, 2):
        for _nm in (True, False):
            CASES.append(_c("terms_%s_norm%d_%s" % (_kern, _norm, "unit" if _nm else "raw"), _kind, 3, 16, 6, 24, 28, tgt=_tgt,
                            norm=_norm, normalize=_nm, terms=ALL_TERMS))
    for _gl in (1.0, 0.37, 0.0):
        CASES.append(_c("qden_gl%g_%s" % (_gl, _kern), _kind, 2, 12, 5, 20, 36, tgt=_tgt, terms=ALL_TERMS, q="x1.7", gl=_gl))
    CASES.append(_c("gm_null_vs_zeros_%s" % _kern, _kind, 2, 12, 5, 20, 36, tgt=_tgt, terms=ALL_TERMS, gm="zeros"))


def _lib():
    from isa_b200 import _lib as L
    return L, L.load()


def _plan(kind, bs, C, K, H, W):
    L, lib = _lib()
    buf = (ctypes.c_int * 12)()
    rc = lib.isa_disc_loss_plan(KINDS[kind], bs, C, K, H, W, buf)
    if rc:
        return rc, None
    keys = "route CP priv lab_G lab_grid lab_smem col_G col_grid col_smem prep_smem bwd_gx bwd_smem".split()
    return 0, dict(zip(keys, list(buf)))


def _inputs(c, dev):
    """-> (emb f32 device, target device, n_objects i32 device, labels numpy or None)."""
    n_max = c.n_max or min(c.K, 23)
    n_min = n_max if c.nobj is not None and max(c.nobj) > c.K else 1     # n_objects above K: every id below K present
    d = synth.batch(CASES.index(c) * 7 + 1 if c in CASES else 99, c.bs, c.C, c.H, c.W, c.K, n_min=n_min, n_max=n_max, pull=0.4)
    lab, nobj = d["labels"].copy(), d["n_objects"].copy()
    rs = np.random.RandomState(c.bs * 1000 + c.C)
    if c.bg in ("image", "batch"):
        lab[0] = 255
        nobj[0] = 0
        if c.bg == "batch":
            lab[:] = 255
            nobj[:] = 0
    if c.hi:
        bgm = lab == 255
        nbg = int(bgm.sum())
        lab[bgm] = np.where(rs.uniform(size=nbg) < 0.5, rs.randint(c.K, 255, size=nbg), 255).astype(np.uint8)
    if c.nobj is not None:
        nobj = np.array(c.nobj, dtype=np.int32)
    emb = torch.tensor(d["emb"], device=dev)
    if c.kind == "label":
        return emb, torch.tensor(lab, device=dev), torch.tensor(nobj, device=dev), lab
    dt = DTYPES[c.kind]
    oh = synth.onehot(lab, c.K, np.float64)
    if c.tgt == "onehot":
        t = oh
    elif c.tgt == "soft":
        t = oh * rs.uniform(0.2, 1.0, size=oh.shape) + (rs.uniform(size=oh.shape) > 0.85) * rs.uniform(size=oh.shape)
    elif c.tgt == "overlap":
        t = oh + (rs.uniform(size=oh.shape) > 0.9) * rs.randint(1, 3, size=oh.shape)
    elif c.tgt == "single_w":
        t = oh.copy()
        b, y, x = [int(v[0]) for v in np.nonzero(lab < 255)]
        t[b, :, y, x] = 0
        t[b, int(nobj[b]) - 1, y, x] = 0.5 if c.kind == "f32" else 3
    else:   # high_ch: a block of pixels with two or more entries, all in channels >= n_objects
        t = oh.copy()
        for b in range(c.bs):
            t[b, :, :4, :6] = 0
            t[b, int(nobj[b]):, :4, :6] = (rs.uniform(size=(c.K - int(nobj[b]), 4, 6)) > 0.3) * 2
    return emb, torch.tensor(t.astype(dt), device=dev), torch.tensor(nobj, device=dev), None


def _guarded(numel, dev):
    store = torch.full((GUARD + numel + GUARD,), SENTINEL, dtype=torch.int32, device=dev)
    return store, store[GUARD:GUARD + numel].view(torch.float32)


def _written(store, what):
    inside = store[GUARD:-GUARD]
    assert not bool((inside == SENTINEL).any()), "%s: %d elements not written" % (what, int((inside == SENTINEL).sum()))
    assert bool((store[:GUARD] == SENTINEL).all() and (store[-GUARD:] == SENTINEL).all()), "%s: written outside the buffer" % what


def _untouched(store, what):
    assert bool((store == SENTINEL).all()), "%s written by a refused call" % what


class Caller(object):
    """Calls isa_disc_loss_fwd / _bwd on one problem with guarded outputs."""

    def __init__(self, c, dev, emb, tgt, nobj):
        self.c, self.dev, self.emb, self.tgt, self.nobj = c, dev, emb, tgt, nobj
        self.kind = KINDS[c.kind]
        L, lib = _lib()
        self.ws_bytes = lib.isa_disc_loss_workspace_bytes(c.bs, c.C, c.K, c.H, c.W)

    def new_ws(self, fill):
        return torch.full((self.ws_bytes,), fill, dtype=torch.uint8, device=self.dev)

    def fwd(self, ws, q_den=None, expect=0):
        L, lib = _lib()
        c = self.c
        s = {k: _guarded(n, self.dev) for k, n in (("loss", 1), ("terms", 4), ("means", c.bs * c.K * c.C))}
        rc = lib.isa_disc_loss_fwd(L.ptr(self.emb), L.ptr(self.tgt), self.kind, L.ptr(self.nobj), c.bs, c.C, c.H, c.W, c.K,
                                   DV, DD, c.norm, int(c.normalize), *c.terms, L.ptr(q_den), L.ptr(s["loss"][1]),
                                   L.ptr(s["terms"][1]), L.ptr(s["means"][1]), L.ptr(ws), self.ws_bytes, L.stream_ptr(self.dev))
        torch.cuda.synchronize()
        assert rc == expect, "isa_disc_loss_fwd: rc %d (%s)" % (rc, lib.isa_last_error())
        for k, (st, _) in s.items():
            (_written if expect == 0 else _untouched)(st, k)
        return {k: v[1].clone().view(torch.float32) for k, v in s.items()}

    def bwd(self, ws, means, gl, gm, q_den=None, expect=0):
        L, lib = _lib()
        c = self.c
        st, g = _guarded(self.emb.numel(), self.dev)
        glt = torch.tensor([gl], dtype=torch.float32, device=self.dev)
        rc = lib.isa_disc_loss_bwd(L.ptr(self.emb), L.ptr(self.tgt), self.kind, L.ptr(self.nobj), c.bs, c.C, c.H, c.W, c.K,
                                   DV, DD, c.norm, int(c.normalize), *c.terms, L.ptr(q_den), L.ptr(means), L.ptr(glt), L.ptr(gm),
                                   L.ptr(g), L.ptr(ws), self.ws_bytes, L.stream_ptr(self.dev))
        torch.cuda.synchronize()
        assert rc == expect, "isa_disc_loss_bwd: rc %d (%s)" % (rc, lib.isa_last_error())
        (_written if expect == 0 else _untouched)(st, "grad_emb")
        return g.clone().view(self.emb.shape)


def _local_fg(tgt, K):
    if tgt.dim() == 3:
        return float(int((tgt < K).sum()))
    return float(int(tgt.double().sum()))


def _check_scalar(a, b, what, rtol=RTOL):
    a, b = float(a), float(b)
    if np.isnan(b) or np.isinf(b):
        assert (np.isnan(a) and np.isnan(b)) or a == b, "%s: %r, reference %r" % (what, a, b)
    else:
        assert abs(a - b) <= rtol * abs(b) + 1e-7, "%s: %r, reference %r (rel %.2e)" % (what, a, b, abs(a - b) / max(abs(b), 1e-30))


def _check_against(out, g, ref, K, nobj, what=""):
    """out / g: the kernel's forward outputs and gradient; ref: oracle/disc_loss_torch.py.  -> worst relative errors."""
    _check_scalar(out["loss"][0], ref["loss"], what + "loss")
    for i, t in enumerate("var dist reg qreg".split()):
        _check_scalar(out["terms"][i], ref["terms"][i], what + "term " + t)
    m, mr = out["means"].view(ref["means"].shape).double(), ref["means"]
    assert torch.equal(torch.isnan(m), torch.isnan(mr)), what + "means: NaN in different places"
    fin = ~torch.isnan(mr)
    merr = float((m[fin] - mr[fin]).abs().max()) if bool(fin.any()) else 0.0
    assert merr <= MEANS_ATOL, "%smeans: max abs error %.3e" % (what, merr)
    for b, n in enumerate(nobj.tolist()):
        assert bool((m[b, max(min(n, K), 0):] == 0).all()), "%smeans rows k >= n_objects of image %d are not 0" % (what, b)
    gd, gr = g.double(), ref["grad"]
    assert torch.equal(torch.isnan(gd), torch.isnan(gr)), "%sgrad: NaN in different places (%d vs %d)" % (
        what, int(torch.isnan(gd).sum()), int(torch.isnan(gr).sum()))
    assert not bool(torch.isinf(gd).any()) and not bool(torch.isinf(gr).any())
    fin = ~torch.isnan(gr)
    scale = max(float(gr[fin].abs().max()) if bool(fin.any()) else 0.0, 1e-30)
    gerr = float((gd[fin] - gr[fin]).abs().max()) / scale if bool(fin.any()) else 0.0
    assert gerr <= GRAD_RTOL, "%sgrad: error %.3e of the largest element" % (what, gerr)
    lref = float(ref["loss"])
    lerr = abs(float(out["loss"][0]) - lref) / abs(lref) if np.isfinite(lref) and lref != 0 else 0.0
    return lerr, merr, gerr


def _same_bits(a, b, what):
    for k in a:
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), "%s: %s differs" % (what, k)


def _ref(c, emb, tgt, nobj, q_den, gl, gm):
    return R.discriminative_loss(emb, tgt, nobj.cpu(), c.K, DV, DD, c.norm, terms=c.terms, normalize_means=c.normalize,
                                 q_den=None if q_den is None else float(q_den), grad_loss=gl,
                                 grad_means=gm, want_grad=True)


@pytest.mark.parametrize("c", CASES, ids=[c.name for c in CASES])
def test_disc_loss_against_float64(cuda, c):
    rc, plan = _plan(c.kind, c.bs, c.C, c.K, c.H, c.W)
    assert rc == 0, "isa_disc_loss_plan: rc %d" % rc
    emb, tgt, nobj, lab = _inputs(c, cuda)
    call = Caller(c, cuda, emb, tgt, nobj)
    q_den = None
    if c.q == "x1.7":
        q_den = torch.tensor([1.7 * _local_fg(tgt, c.K)], dtype=torch.float32, device=cuda)
    gm = None
    if c.gm == "rand":
        gm = torch.randn(c.bs, c.K, c.C, generator=torch.Generator(device=cuda).manual_seed(5), device=cuda) * 0.01

    ws = call.new_ws(0xFF)
    out = call.fwd(ws, q_den)
    g = call.bwd(ws, out["means"], c.gl, gm, q_den)
    ref = _ref(c, emb, tgt, nobj, q_den, c.gl, gm)
    errs = _check_against(out, g, ref, c.K, nobj)
    print("%s: route %s priv %d CP %d; loss rel %.2e, means abs %.2e, grad rel %.2e"
          % (c.name, ROUTE_NAMES[plan["route"]], plan["priv"], plan["CP"], *errs))

    # the forward zeroes what it relies on: a zeroed workspace gives the same result
    ws0 = call.new_ws(0)
    out0 = call.fwd(ws0, q_den)
    g0 = call.bwd(ws0, out0["means"], c.gl, gm, q_den)
    deterministic = plan["route"] == ROUTE_LAB or (plan["route"] == ROUTE_COL_THEN_LAB and c.tgt == "onehot")
    deterministic = deterministic and plan["priv"] == 1
    if deterministic:
        _same_bits(out0, out, c.name + ": 0xFF vs zeroed workspace")
        assert torch.equal(g0.view(torch.int32), g.view(torch.int32)), "backward differs between two runs"
    else:
        _check_against(out0, g0, ref, c.K, nobj, "zeroed workspace: ")

    if c.q == "local":        # q_den equal to the local count: the same bits as NULL
        qd = torch.tensor([_local_fg(tgt, c.K)], dtype=torch.float32, device=cuda)
        ws1 = call.new_ws(0xFF)
        out1 = call.fwd(ws1, qd)
        g1 = call.bwd(ws1, out1["means"], c.gl, gm, qd)
        if deterministic:
            _same_bits(out1, out, "q_den = local count vs NULL")
            assert torch.equal(g1.view(torch.int32), g.view(torch.int32)), "q_den = local count vs NULL: grad differs"
        _check_against(out1, g1, ref, c.K, nobj, "q_den = local count: ")
    if c.gm == "zeros":       # grad_means of zeros: the same bits as NULL (same forward workspace)
        assert gm is None
        gz = call.bwd(ws, out["means"], c.gl, torch.zeros(c.bs, c.K, c.C, device=cuda))
        assert torch.equal(gz.view(torch.int32), g.view(torch.int32)), "grad_means zeros vs NULL: grad differs"
    if c.kind != "label" and c.tgt == "onehot":   # a dense one-hot target runs the same kernels as its label map
        lab_t = torch.where((tgt != 0).any(1), tgt.double().argmax(1), torch.full_like(tgt[:, 0], 255, dtype=torch.int64)).to(torch.uint8)
        cl = Caller(c._replace(kind="label"), cuda, emb, lab_t.contiguous(), nobj)
        wsl = cl.new_ws(0xFF)
        outl = cl.fwd(wsl, q_den)
        gl_ = cl.bwd(wsl, outl["means"], c.gl, gm, q_den)
        if deterministic:
            _same_bits(outl, out, "dense one-hot vs label map")
            assert torch.equal(gl_.view(torch.int32), g.view(torch.int32)), "dense one-hot vs label map: grad differs"
        else:
            _check_against(outl, gl_, ref, c.K, nobj, "label map of the one-hot target: ")


def test_cases_reach_every_route(cuda):
    seen = []
    for c in CASES:
        rc, p = _plan(c.kind, c.bs, c.C, c.K, c.H, c.W)
        assert rc == 0, c.name
        seen.append((c, p))
    missing = []

    def need(what, pred):
        if not any(pred(c, p) for c, p in seen):
            missing.append(what)

    for CP in (8, 16, 24, 32, 64):
        need("lab priv=1 CP=%d, several CTAs per image" % CP,
             lambda c, p: p["route"] == ROUTE_LAB and p["priv"] == 1 and p["CP"] == CP and p["lab_G"] > 1)
        need("lab priv=1 CP=%d, one CTA per image" % CP,
             lambda c, p: p["route"] == ROUTE_LAB and p["priv"] == 1 and p["CP"] == CP and p["lab_G"] == 1)
    need("lab priv=0", lambda c, p: p["route"] == ROUTE_LAB and p["priv"] == 0)
    need("col on a label map, looping over images",
         lambda c, p: p["route"] == ROUTE_COL and c.kind == "label" and p["col_grid"] < c.bs)
    need("col on a label map, bs above 640", lambda c, p: p["route"] == ROUTE_COL and c.kind == "label" and c.bs > 640)
    for k in ("f32", "i64", "u8"):
        need("col on the label map distilled from a one-hot %s target" % k,
             lambda c, p: p["route"] == ROUTE_COL and c.kind == k and c.tgt == "onehot" and p["col_grid"] < c.bs)
        need("col early exit then lab, one-hot %s" % k,
             lambda c, p: p["route"] == ROUTE_COL_THEN_LAB and c.kind == k and c.tgt == "onehot")
        need("col on %s masks that are not one-hot, several CTAs per image" % k,
             lambda c, p: p["route"] == ROUTE_COL_THEN_LAB and c.kind == k and c.tgt != "onehot" and p["col_G"] > 1)
    need("col on soft masks, looping over images",
         lambda c, p: p["route"] != ROUTE_LAB and c.tgt == "soft" and p["col_grid"] < c.bs)
    need("col at CP=64", lambda c, p: p["route"] != ROUTE_LAB and c.tgt != "onehot" and p["CP"] == 64)
    need("an image of fewer than 256 pixels with W < 32", lambda c, p: c.H * c.W < 256 and c.W < 32)
    need("an image with H = 1", lambda c, p: c.H == 1)
    need("an image with W = 1", lambda c, p: c.W == 1)
    routes = sorted(set(ROUTE_NAMES[p["route"]] for _, p in seen))
    print("routes reached: %s" % ", ".join(routes))
    assert not missing, "routes no case reaches: %s" % "; ".join(missing)


def test_workspace_reused_for_another_batch(cuda):
    """One workspace, two batches of the same shape: the second result equals a fresh-workspace run bit for bit.
    The first batch is soft masks (not one-hot), the second one-hot: the flag left in the workspace must not matter."""
    c = _c("reuse", "f32", 3, 16, 8, 30, 40)
    emb, tgt, nobj, _ = _inputs(c, cuda)
    soft = _c("reuse_soft", "f32", 3, 16, 8, 30, 40, tgt="soft")
    emb2, tgt2, nobj2, _ = _inputs(soft, cuda)
    first = Caller(soft, cuda, emb2 * 1.3, tgt2, nobj2)
    second = Caller(c, cuda, emb, tgt, nobj)
    ws = first.new_ws(0xFF)
    o = first.fwd(ws)
    first.bwd(ws, o["means"], 1.0, None)
    out = second.fwd(ws)
    g = second.bwd(ws, out["means"], 1.0, None)
    wsf = second.new_ws(0xFF)
    outf = second.fwd(wsf)
    gf = second.bwd(wsf, outf["means"], 1.0, None)
    _same_bits(out, outf, "reused vs fresh workspace")
    assert torch.equal(g.view(torch.int32), gf.view(torch.int32)), "reused vs fresh workspace: grad differs"


def test_limits_at_C64_K254(cuda):
    """C = 64, K = 254, the largest the header accepts.  The label-map kernel fits (priv = 0), with a backward whose prep
    kernel needs 65,024 B of shared memory.  The column walk needs more than an SM has: a dense target, or a label map
    with bs above the label-map kernel's co-resident CTAs, is refused before anything is enqueued."""
    rc, p = _plan("label", 2, 64, 254, 24, 24)
    assert rc == 0 and p["route"] == ROUTE_LAB and p["priv"] == 0 and p["prep_smem"] == 4 * 254 * 64
    c = _c("C64_K254_label", "label", 2, 64, 254, 24, 24, n_max=200, terms=ALL_TERMS)
    emb, tgt, nobj, _ = _inputs(c, cuda)
    call = Caller(c, cuda, emb, tgt, nobj)
    ws = call.new_ws(0xFF)
    out = call.fwd(ws)
    g = call.bwd(ws, out["means"], 1.0, None)
    _check_against(out, g, _ref(c, emb, tgt, nobj, None, 1.0, None), c.K, nobj)

    # the smallest of these batch sizes above the label-map kernel's co-resident CTAs (148 on a B200 at this size)
    lab_cap = next((bs for bs in (149, 297, 641) if _plan("label", bs, 64, 254, 2, 2)[0] == ISA_ERR_UNSUPPORTED), None)
    assert lab_cap is not None
    for name, kind, bs, H, W in (("dense one-hot", "i64", 2, 8, 8), ("label map, bs above the co-resident CTAs", "label", lab_cap, 2, 2)):
        rc, _ = _plan(kind, bs, 64, 254, H, W)
        assert rc == ISA_ERR_UNSUPPORTED, "%s: plan rc %d" % (name, rc)
        c = _c("C64_K254", kind, bs, 64, 254, H, W, n_max=2)
        emb, tgt, nobj, _ = _inputs(c, cuda)
        call = Caller(c, cuda, emb, tgt, nobj)
        ws = torch.full((call.ws_bytes // 4 + 1,), SENTINEL, dtype=torch.int32, device=cuda)
        call.fwd(ws, expect=ISA_ERR_UNSUPPORTED)
        assert bool((ws == SENTINEL).all()), "%s: workspace written by a refused forward" % name
    # the largest K that fits at C = 64 runs the column walk (soft_C64_K213 checks its result); one more does not
    assert _plan("f32", 2, 64, 213, 8, 8)[0] == 0 and _plan("f32", 2, 64, 214, 8, 8)[0] == ISA_ERR_UNSUPPORTED


def test_rejects_bad_arguments(cuda):
    """Each bad argument is refused before anything is enqueued: outputs and workspace keep their sentinel."""
    L, lib = _lib()
    st = L.stream_ptr(cuda)
    bs, C, H, W, K = 2, 8, 6, 7, 4
    emb = torch.randn(bs, C, H, W, device=cuda)
    tgt = torch.zeros(bs, H, W, dtype=torch.uint8, device=cuda)
    nobj = torch.ones(bs, dtype=torch.int32, device=cuda)
    means_in = torch.randn(bs, K, C, device=cuda)
    glt = torch.ones(1, device=cuda)
    ws_bytes = lib.isa_disc_loss_workspace_bytes(bs, C, K, H, W)
    outs = {k: _guarded(n, cuda) for k, n in (("loss", 1), ("terms", 4), ("means", bs * K * C), ("grad", emb.numel()),
                                              ("ws", ws_bytes // 4 + 1))}
    P = L.ptr
    o = {k: P(v[1]) for k, v in outs.items()}

    def fwd(**kw):
        a = dict(emb=P(emb), tgt=P(tgt), kind=0, nobj=P(nobj), bs=bs, C=C, H=H, W=W, K=K, norm=2, loss=o["loss"], terms=o["terms"],
                 means=o["means"], ws=o["ws"], ws_bytes=ws_bytes)
        a.update(kw)
        return lib.isa_disc_loss_fwd(a["emb"], a["tgt"], a["kind"], a["nobj"], a["bs"], a["C"], a["H"], a["W"], a["K"], DV, DD,
                                     a["norm"], 1, *SHIPPED, None, a["loss"], a["terms"], a["means"], a["ws"], a["ws_bytes"], st)

    def bwd(**kw):
        a = dict(emb=P(emb), tgt=P(tgt), kind=0, nobj=P(nobj), bs=bs, C=C, H=H, W=W, K=K, norm=2, means=P(means_in), gl=P(glt),
                 grad=o["grad"], ws=o["ws"], ws_bytes=ws_bytes)
        a.update(kw)
        return lib.isa_disc_loss_bwd(a["emb"], a["tgt"], a["kind"], a["nobj"], a["bs"], a["C"], a["H"], a["W"], a["K"], DV, DD,
                                     a["norm"], 1, *SHIPPED, None, a["means"], a["gl"], None, a["grad"], a["ws"], a["ws_bytes"], st)

    bad = [dict(kind=4), dict(kind=-1), dict(C=0), dict(C=65), dict(K=0), dict(K=255), dict(norm=0), dict(norm=3), dict(bs=0),
           dict(H=1 << 15, W=1 << 15), dict(H=0)]
    calls = [("fwd", kw, fwd, ISA_ERR_BAD_ARG) for kw in bad + [dict(emb=None), dict(tgt=None), dict(nobj=None), dict(loss=None),
                                                                 dict(terms=None), dict(means=None), dict(ws=None)]]
    calls += [("bwd", kw, bwd, ISA_ERR_BAD_ARG) for kw in bad + [dict(emb=None), dict(tgt=None), dict(nobj=None), dict(means=None),
                                                                  dict(gl=None), dict(grad=None), dict(ws=None)]]
    calls += [(pas, dict(ws_bytes=ws_bytes - 1), fn, ISA_ERR_WORKSPACE) for pas, fn in (("fwd", fwd), ("bwd", bwd))]
    for pas, kw, fn, want in calls:
        rc = fn(**kw)
        assert rc == want, "%s %s: rc %d" % (pas, kw, rc)
        assert b"disc_loss" in lib.isa_last_error(), (pas, kw)
    buf = (ctypes.c_int * 12)()
    for kw in bad:
        a = dict(kind=0, bs=bs, C=C, K=K, H=H, W=W)
        a.update({k: v for k, v in kw.items() if k in a})
        if "norm" in kw:
            continue
        assert lib.isa_disc_loss_plan(a["kind"], a["bs"], a["C"], a["K"], a["H"], a["W"], buf) == ISA_ERR_BAD_ARG, kw
    torch.cuda.synchronize()
    for name, (store, _) in outs.items():
        _untouched(store, name)


def test_backward_refuses_bs_above_65535_before_enqueuing(cuda):
    """The backward's grid has one row per image (at most 65535): a larger batch is refused with the workspace as it was."""
    L, lib = _lib()
    bs, C, K = 65536, 1, 1
    emb = torch.randn(bs, C, 1, 1, device=cuda)
    tgt = torch.zeros(bs, 1, 1, dtype=torch.uint8, device=cuda)
    nobj = torch.ones(bs, dtype=torch.int32, device=cuda)
    means = torch.randn(bs, K, C, device=cuda)
    glt = torch.ones(1, device=cuda)
    ws_bytes = lib.isa_disc_loss_workspace_bytes(bs, C, K, 1, 1)
    ws_s, ws = _guarded(ws_bytes // 4 + 1, cuda)
    g_s, g = _guarded(emb.numel(), cuda)
    rc = lib.isa_disc_loss_bwd(L.ptr(emb), L.ptr(tgt), 0, L.ptr(nobj), bs, C, 1, 1, K, DV, DD, 2, 1, *SHIPPED, None, L.ptr(means),
                               L.ptr(glt), None, L.ptr(g), L.ptr(ws), ws_bytes, L.stream_ptr(cuda))
    torch.cuda.synchronize()
    assert rc == ISA_ERR_BAD_ARG
    _untouched(ws_s, "workspace")
    _untouched(g_s, "grad_emb")


def test_foreground_counts(cuda):
    """isa_onehot_to_labels' fg_count and isa_label_fg_count against numpy, with K below the largest label."""
    from isa_b200.losses import label_fg_count, onehot_to_labels
    d = synth.batch(31, 3, 4, 33, 47, 16, n_min=10, n_max=16)
    lab = d["labels"].copy()
    lab[0, :3] = 200
    for K in (16, 5, 1, 254):
        cnt = label_fg_count(torch.tensor(lab, device=cuda), K)
        assert int(cnt) == int((lab < K).sum()), K
    for dt in (np.float32, np.int64, np.uint8):
        oh = synth.onehot(d["labels"], 16, dt)
        labels, flag, cnt = onehot_to_labels(torch.tensor(oh, device=cuda), with_count=True)
        assert int(cnt) == int((d["labels"] < 16).sum()) and int(flag) == 0
        assert np.array_equal(labels.cpu().numpy(), d["labels"])
        # the flag and the count when a pixel is not one-hot: the count is of pixels with any non-zero entry
        oh2 = oh.copy()
        oh2[1, 3, 0, 0] = 2
        oh2[2, :2, 5, 5] = 1
        _, flag, cnt = onehot_to_labels(torch.tensor(oh2, device=cuda), with_count=True)
        assert int(flag) == 1 and int(cnt) == int((oh2 != 0).any(1).sum())


@pytest.mark.parametrize("kind", ["label", "i64"])
def test_full_size_against_float64(cuda, kind):
    """The bench's train step (bs 16, C 24, K 32, 256 x 256) through DiscriminativeLoss, against the float64 reference."""
    from isa_b200.losses import DiscriminativeLoss
    d = synth.batch(123, 16, 24, 256, 256, 32)
    x = torch.tensor(d["emb"], device=cuda, requires_grad=True)
    lab = torch.tensor(d["labels"], device=cuda)
    n = torch.tensor(d["n_objects"], device=cuda)
    tgt = lab if kind == "label" else torch.tensor(synth.onehot(d["labels"], 32, np.int64), device=cuda)
    crit = DiscriminativeLoss(DV, DD, 2)
    loss, means = crit(x, tgt, n, 32)
    loss.backward()
    ref = R.discriminative_loss(x.detach(), lab, d["n_objects"], 32, DV, DD, 2, want_grad=True)
    lerr, merr, gerr = _check_against(dict(loss=loss.detach().reshape(1), terms=crit.last_terms, means=means.detach()),
                                      x.grad, ref, 32, n)
    print("full size %s: loss rel %.2e, means abs %.2e, grad rel %.2e" % (kind, lerr, merr, gerr))


def test_data_parallel_rank_against_float64(cuda):
    """One rank of the two-GPU run: bs 8 with q_den = global foreground / 2, against the float64 reference."""
    from isa_b200.losses import DiscriminativeLoss
    d = synth.batch(321, 16, 24, 256, 256, 32)
    global_fg = int((d["labels"] < 32).sum())
    q_den = torch.tensor([global_fg / 2.0], dtype=torch.float32, device=cuda)
    x = torch.tensor(d["emb"][:8], device=cuda, requires_grad=True)
    lab = torch.tensor(d["labels"][:8], device=cuda)
    n = torch.tensor(d["n_objects"][:8], device=cuda)
    crit = DiscriminativeLoss(DV, DD, 2)
    loss, means = crit(x, lab, n, 32, q_denominator=q_den)
    loss.backward()
    ref = R.discriminative_loss(x.detach(), lab, d["n_objects"][:8], 32, DV, DD, 2, q_den=float(q_den), want_grad=True)
    _check_against(dict(loss=loss.detach().reshape(1), terms=crit.last_terms, means=means.detach()), x.grad, ref, 32, n)
