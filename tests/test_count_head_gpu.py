"""GPU: the instance-count head -- the fused tail kernels (isa_count_head_fwd / _bwd) over every shape class against the
float64 oracle (oracle/count_head_ref.py), the wired branch of ReSeg(count_head=True), the training step with the count
loss (eager, CUDA graph, data-parallel identity), and prediction with per-image predicted counts."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from isa_b200 import _lib, synth
from oracle import count_head_ref as CH
from oracle import kmeans as KM

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GUARD = 4                      # 16 bytes: keeps the guarded buffers 16-byte aligned
SENT = -777777


def _guarded(n, dtype, dev, fill):
    buf = torch.full((n + 2 * GUARD,), fill, dtype=dtype, device=dev)
    return buf, buf[GUARD:GUARD + n]


def _guards_intact(buf, fill):
    g = torch.cat([buf[:GUARD], buf[-GUARD:]])
    return bool(torch.isnan(g).all()) if buf.dtype.is_floating_point else bool((g == fill).all())


class _Tail(object):
    """Guarded buffers of one forward + backward call."""

    def __init__(self, x, conv_bias, w, b, nobj, K, dev):
        self.bs, self.P, self.C = x.shape
        self.K = K
        bs, P, C = x.shape
        self.xb, self.x = _guarded(bs * P * C, torch.float32, dev, float("nan"))
        self.x.copy_(x.reshape(-1))
        self.conv_bias, self.w, self.b = conv_bias, w, b
        self.nobj = nobj
        self.pb, self.pooled = _guarded(bs * C, torch.float32, dev, float("nan"))
        self.sb, self.s = _guarded(bs, torch.float32, dev, float("nan"))
        self.nb, self.n_pred = _guarded(bs, torch.int32, dev, SENT)
        self.lb, self.loss = _guarded(1, torch.float32, dev, float("nan"))
        self.gb, self.gx = _guarded(bs * P * C, torch.float32, dev, float("nan"))
        self.dcb_b, self.dcb = _guarded(C, torch.float32, dev, float("nan"))
        self.dwb, self.dw = _guarded(C, torch.float32, dev, float("nan"))
        self.dbb, self.db = _guarded(1, torch.float32, dev, float("nan"))
        self.wsb = _lib.load().isa_count_head_workspace_bytes(bs, P, C)
        self.ws = torch.empty(self.wsb, dtype=torch.uint8, device=dev)

    def fwd(self, with_loss=True, **over):
        a = dict(x=self.x.data_ptr(), conv_bias=self.conv_bias.data_ptr(), w=self.w.data_ptr(), b=self.b.data_ptr(),
                 n_objects=self.nobj.data_ptr() if with_loss else None, bs=self.bs, P=self.P, C=self.C, K=self.K,
                 pooled=self.pooled.data_ptr(), s=self.s.data_ptr(), n_pred=self.n_pred.data_ptr(),
                 loss=self.loss.data_ptr() if with_loss else None, ws=self.ws.data_ptr(), wsb=self.wsb)
        a.update(over)
        return _lib.load().isa_count_head_fwd(*a.values(), _lib.stream_ptr())

    def bwd(self, gl, **over):
        a = dict(y=self.x.data_ptr(), pooled=self.pooled.data_ptr(), s=self.s.data_ptr(), w=self.w.data_ptr(),
                 n_objects=self.nobj.data_ptr(), grad_loss=gl.data_ptr(), bs=self.bs, P=self.P, C=self.C, K=self.K,
                 gx=self.gx.data_ptr(), dcb=self.dcb.data_ptr(), dw=self.dw.data_ptr(), db=self.db.data_ptr(),
                 ws=self.ws.data_ptr(), wsb=self.wsb)
        a.update(over)
        return _lib.load().isa_count_head_bwd(*a.values(), _lib.stream_ptr())

    def guards_intact(self):
        return all(_guards_intact(b, SENT) for b in (self.xb, self.pb, self.sb, self.nb, self.lb, self.gb, self.dcb_b,
                                                      self.dwb, self.dbb))


def _inputs(bs, P, C, K, case, dev):
    g = torch.Generator().manual_seed(1000 * bs + 10 * C + K + P)
    x = torch.randn(bs, P, C, generator=g, dtype=torch.float64) - 0.2
    x[:, :, 1] = -2.0 - torch.rand(bs, P, generator=g, dtype=torch.float64)   # ReLU kills channel 1 everywhere
    conv_bias = 0.1 * torch.randn(C, generator=g, dtype=torch.float64)
    w = torch.randn(C, generator=g, dtype=torch.float64) / C ** 0.5
    b = torch.tensor([(0.1, 40.0, -40.0)[case % 3]], dtype=torch.float64)          # case 1, 2: saturated sigmoids
    nobj = torch.randint(0, K + 1, (bs,), generator=g, dtype=torch.int32)
    nobj[0] = 0
    nobj[-1] = K
    f = lambda t: t.float().to(dev)
    return x, conv_bias, w, b, nobj, (f(x), f(conv_bias), f(w), f(b), nobj.to(dev))


def _close(got, want, rel):
    got, want = got.double().cpu(), want.double().cpu()
    return float((got - want).abs().max()) <= rel * max(float(want.abs().max()), 1e-30) + 1e-12


SHAPES = [(bs, P, C) for bs in (1, 3, 16, 17) for P in (1, 7, 256, 4097, 8192) for C in (4, 64, 256)]


@pytest.mark.parametrize("bs,P,C", SHAPES)
def test_tail_kernels_match_float64_oracle(cuda, bs, P, C):
    i = SHAPES.index((bs, P, C))
    K = (1, 32, 64)[(i + i // 3) % 3]          # every (C, K) pair occurs
    x, cb, w, b, nobj, (xf, cbf, wf, bf, nobj_d) = _inputs(bs, P, C, K, i // 3, cuda)
    t = _Tail(xf, cbf, wf, bf, nobj_d, K, cuda)
    assert t.fwd() == 0
    gl = torch.tensor([0.75], device=cuda)
    assert t.bwd(gl) == 0
    torch.cuda.synchronize()
    assert t.guards_intact()
    # oracle in float64 from the same float32 inputs
    x64, cb64, w64, b64 = xf.double(), cbf.double(), wf.double(), bf.double()
    y = torch.relu(x64 + cb64).permute(0, 2, 1).reshape(bs, C, 1, P)          # NCHW view of the NHWC map
    pooled, s = CH.tail(y, w64, b64)
    loss = CH.count_loss(s, nobj_d, K)
    gx, dcb, dw, db = CH.tail_grad(y, pooled, s, w64, nobj_d, K, grad_loss=0.75)
    ky = t.x.view(bs, P, C)
    assert _close(ky, y.reshape(bs, C, P).permute(0, 2, 1), 1e-5)
    assert _close(t.pooled.view(bs, C), pooled, 1e-5)
    assert float(((t.s.double() - s).abs() / s.abs().clamp_min(1e-300)).max()) <= 1e-5
    assert abs(float(t.loss[0]) - float(loss)) <= 1e-5
    assert torch.equal(t.n_pred.cpu(), torch.round(t.s * K).clamp(1, K).to(torch.int32).cpu())
    assert _close(t.gx.view(bs, P, C), gx.reshape(bs, C, P).permute(0, 2, 1), 1e-4)
    for got, want in ((t.dcb, dcb), (t.dw, dw), (t.db, db)):
        assert _close(got, want, 1e-4)
    for buf in (t.x, t.pooled, t.s, t.loss, t.gx, t.dcb, t.dw, t.db):       # every element written
        assert bool(torch.isfinite(buf).all())
    if bs * P * C <= 3 * 4097 * 64:
        # repeated calls: identical bits (the in-place forward is rerun on the same pre-activation)
        first = [u.clone() for u in (t.x, t.pooled, t.s, t.n_pred, t.loss, t.gx, t.dcb, t.dw, t.db)]
        t.x.copy_(xf.reshape(-1))
        assert t.fwd() == 0 and t.bwd(gl) == 0
        for u, v in zip(first, (t.x, t.pooled, t.s, t.n_pred, t.loss, t.gx, t.dcb, t.dw, t.db)):
            assert torch.equal(u, v)
        # inference call: no targets, no loss; the same pooled / s / n_pred, the loss buffer untouched
        t.x.copy_(xf.reshape(-1))
        t.lb.fill_(float("nan"))
        assert t.fwd(with_loss=False) == 0
        torch.cuda.synchronize()
        assert torch.equal(t.pooled, first[1]) and torch.equal(t.s, first[2]) and torch.equal(t.n_pred, first[3])
        assert bool(torch.isnan(t.lb).all())


def test_tail_rejects_bad_arguments(cuda):
    bs, P, C, K = 3, 7, 64, 32
    _, _, _, _, _, (xf, cbf, wf, bf, nobj) = _inputs(bs, P, C, K, 0, cuda)
    t = _Tail(xf, cbf, wf, bf, nobj, K, cuda)
    gl = torch.tensor([1.0], device=cuda)
    before = t.x.clone()
    bad_fwd = [dict(C=6), dict(C=260), dict(K=0), dict(K=255), dict(bs=0), dict(P=0), dict(x=None), dict(conv_bias=None),
               dict(w=None), dict(b=None), dict(pooled=None), dict(s=None), dict(n_pred=None), dict(ws=None),
               dict(n_objects=None)]          # the last one: a loss without targets
    for over in bad_fwd:
        assert t.fwd(**over) == -1, over
    bad_bwd = [dict(C=6), dict(C=260), dict(K=0), dict(K=255), dict(bs=0), dict(P=0), dict(y=None), dict(pooled=None),
               dict(s=None), dict(w=None), dict(n_objects=None), dict(grad_loss=None), dict(gx=None), dict(dcb=None),
               dict(dw=None), dict(db=None), dict(ws=None)]
    for over in bad_bwd:
        assert t.bwd(gl, **over) == -1, over
    assert t.fwd(wsb=t.wsb - 1) == -3 and t.bwd(gl, wsb=t.wsb - 1) == -3
    torch.cuda.synchronize()
    assert torch.equal(t.x, before)
    for buf in (t.pooled, t.s, t.loss, t.gx, t.dcb, t.dw, t.db):
        assert bool(torch.isnan(buf).all())
    assert bool((t.n_pred == SENT).all())
    assert t.guards_intact()


# ------------------------------------------------------------------ the wired branch

def _no_tf32_deterministic():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic)
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = False, False, True
    return old


def _restore(old):
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.benchmark, torch.backends.cudnn.deterministic = old


def test_reseg_count_branch_matches_float64_oracle(cuda):
    from isa_b200.archs import ReSeg
    old = _no_tf32_deterministic()
    try:
        torch.manual_seed(4)
        K = 32
        net = ReSeg(2, n_units=20, count_head=True, max_n_objects=K).to(cuda).to(memory_format=torch.channels_last)
        ref = CH.CountBranchRef(2 * 20 + 24).double()
        ref.load_state_dict({k: v.double().cpu() for k, v in net.state_dict().items() if k.startswith("ins_cls")})
        x = torch.randn(2, 3, 64, 64, device=cuda).contiguous(memory_format=torch.channels_last)
        nobj = torch.tensor([3, 9], device=cuda)
        seen = {}
        h = net.path.register_forward_hook(lambda m, i, o: seen.__setitem__("y", o))
        sem, emb, count = net(True, x)
        h.remove()
        out = count.evaluate(nobj)
        out.loss.backward()
        y = seen["y"].detach().double().cpu()
        f, pooled, s = ref(y)
        loss = CH.count_loss(s, nobj.cpu(), K)
        loss.backward()
        assert _close(out.y, f, 5e-4)
        assert _close(out.pooled, pooled, 5e-4)
        assert _close(out.s, s, 5e-4)
        assert abs(float(out.loss) - float(loss)) <= 5e-4 * float(loss)
        assert torch.equal(out.n_pred.cpu(), torch.round(out.s * K).clamp(1, K).int().cpu())
        refp = dict(ref.named_parameters())
        for name, p in net.named_parameters():
            if name.startswith("ins_cls"):
                assert _close(p.grad, refp[name].grad, 5e-4), name
        # the embedding and semantic outputs are those of a head-less network with the same shared weights
        plain = ReSeg(2, n_units=20).to(cuda).to(memory_format=torch.channels_last)
        plain.load_state_dict({k: v for k, v in net.state_dict().items() if not k.startswith("ins_cls")})
        for training in (True, False):
            with torch.set_grad_enabled(training):
                a = net(training, x)
                b = plain(training, x)
            assert len(a) == 3 and len(b) == 2
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    finally:
        _restore(old)


def _count_model(cuda, K=32, seed=23):
    from isa_b200.model import Model
    torch.manual_seed(seed)
    return Model('CVPPP', 'ReSeg', 2, K, use_instance_segmentation=True, n_embedding=24, device=cuda, count_head=True)


def _train_batch(seed, bs, cuda):
    d = synth.batch(seed, bs, 3, 64, 64, 32, n_min=2, n_max=8)
    return [torch.tensor(d["emb"], device=cuda),
            torch.tensor(np.stack([(d["labels"] == 255), (d["labels"] != 255)], 1).astype(np.int64), device=cuda),
            torch.tensor(synth.onehot(d["labels"], 32, np.int64), device=cuda),
            torch.tensor(d["n_objects"], device=cuda)]


def test_count_head_training_lowers_count_cost(cuda):
    m = _count_model(cuda)
    m.define_criterion(None, 0.5, 1.5, 2, False, 'Multi')
    m.define_optimizer(1.0, 0.001, 0.5, 25, 'Adadelta')
    b = _train_batch(7, 4, cuda)
    assert len(set(b[3].tolist())) > 1
    hist = []
    for _ in range(12):
        out = m.train_step(b[0], b[1], b[2], b[3], 10.0)
        hist.append({k: float(v) for k, v in out.items()})
    for h in hist:
        assert all(np.isfinite(v) for v in h.values()), h
        assert set(h) >= {'Cost', 'INS Cost', 'CE Cost', 'Dice Cost', 'Count Cost', 'Count |DiC|'}
    assert hist[-1]['Count Cost'] < hist[0]['Count Cost'], [h['Count Cost'] for h in hist]


def test_count_head_cuda_graph_replay_equals_eager(cuda):
    batches = [_train_batch(seed, 2, cuda) for seed in (5, 6)]
    runs = []
    for graph in (False, True):
        m = _count_model(cuda)
        m.define_criterion(None, 0.5, 1.5, 2, False, 'Multi')
        m.define_optimizer(1.0, 0.001, 0.5, 25, 'Adadelta')
        if graph:
            m.enable_cuda_graph(warmup_steps=2)
        costs, counts = [], []
        for i in range(6):
            b = batches[i % 2]
            out = m.train_step(b[0], b[1], b[2], b[3], 10.0)
            costs.append(float(out['Cost']))
            counts.append(float(out['Count Cost']))
        if graph:
            assert len(m._graphs) == 1
        runs.append((costs, counts, torch.cat([p.detach().reshape(-1) for p in m.model.parameters()]).clone()))
    (c0, k0, p0), (c1, k1, p1) = runs
    assert c1[0] == c0[0], (c1[0], c0[0])
    np.testing.assert_allclose(c1, c0, rtol=2e-4)
    np.testing.assert_allclose(k1, k0, rtol=2e-4)
    assert _close(p1, p0, 1e-3)


def test_count_loss_data_parallel_identity(cuda):
    """Equal shards, averaged gradients: the per-shard batch mean of the count loss gives the full-batch gradient."""
    old = _no_tf32_deterministic()
    try:
        m = _count_model(cuda)
        m.model.train(True)
        b = _train_batch(8, 4, cuda)
        images = b[0].contiguous(memory_format=torch.channels_last)
        params = [p for n, p in m.model.named_parameters()]

        def grads(sl):
            loss = m.model(True, images[sl])[2].evaluate(b[3][sl]).loss
            g = torch.autograd.grad(loss, params, allow_unused=True)
            return torch.cat([(gi if gi is not None else torch.zeros_like(p)).reshape(-1) for gi, p in zip(g, params)])

        full = grads(slice(0, 4))
        avg = 0.5 * (grads(slice(0, 2)) + grads(slice(2, 4)))
        assert float(full.abs().max()) > 0
        assert _close(avg, full, 1e-5)
    finally:
        _restore(old)


# ------------------------------------------------------------------ prediction with predicted counts

def _prediction(cuda, strict=True):
    from isa_b200.prediction import Prediction
    from isa_b200.settings import CVPPPModelSettings
    ms = CVPPPModelSettings()
    m = _count_model(cuda, seed=3)
    return m, Prediction(64, 64, ms.MEAN, ms.STD, False, m, 1, seed=0, n_init=4, strict=strict)


def _set_counts(m, pred, raws, counts):
    """Linear layer of the count head solved so that image i predicts counts[i] (min-norm solution of 4 equations)."""
    K = m.max_n_objects
    feats = []
    with torch.no_grad():
        for raw in raws:
            image, _, _ = pred.image_to_tensor(raw)
            x = image.unsqueeze(0).to(m.device).contiguous(memory_format=torch.channels_last)
            feats.append(m.model(False, x)[2].evaluate().pooled[0].double().cpu())
    A = torch.cat([torch.stack(feats), torch.ones(len(raws), 1, dtype=torch.float64)], 1)
    s = torch.tensor(counts, dtype=torch.float64) / K
    z = torch.log(s / (1 - s))
    sol = torch.linalg.lstsq(A, z.reshape(-1, 1), driver="gelsd").solution.reshape(-1)
    lin = m.model.ins_cls_out.linear
    with torch.no_grad():
        lin.weight.copy_(sol[:-1].float().reshape(1, -1))
        lin.bias.copy_(sol[-1:].float())


def test_predict_array_clusters_with_the_predicted_count(cuda):
    m, pred = _prediction(cuda)
    raw = synth.leaf_image(2, 133, 125)
    _set_counts(m, pred, [raw], [5])
    image, h, w = pred.image_to_tensor(raw)
    sem_p, emb, n_pred = m.predict_device_with_counts(image.unsqueeze(0))
    k = int(n_pred[0])
    assert n_pred.dtype == torch.int32 and n_pred.shape == (1,) and k == 5
    assert len(m.predict_device(image.unsqueeze(0))) == 2
    sem_seg, ins_seg, n = pred.predict_array(raw)
    assert n == k
    fg, X = KM.gather_foreground(sem_p[0].cpu().numpy(), emb[0].cpu().numpy())
    assert len(X) >= k
    o = KM.kmeans_oracle(X, k, seed=0, n_init=4)
    assert np.array_equal(ins_seg, KM.upsample_nearest(KM.scatter_labels(fg, o["labels"]), h, w))
    assert np.array_equal(sem_seg, KM.upsample_nearest(fg, h, w))
    _, _, n_t = m.predict(image.unsqueeze(0))
    assert n_t.tolist() == [[k]]


def test_predict_many_with_counts_equals_predict_array(cuda):
    m, pred = _prediction(cuda, strict=False)
    raws = [synth.leaf_image(s, 90 + 7 * s, 80 + 5 * s) for s in range(4)]
    _set_counts(m, pred, raws, [3, 5, 7, 9])
    many = list(pred.predict_many(iter(raws)))
    assert len(many) == len(raws)
    ns = []
    for raw, (sem, ins, n) in zip(raws, many):
        sem1, ins1, n1 = pred.predict_array(raw)
        assert n == n1 and np.array_equal(sem, sem1) and np.array_equal(ins, ins1)
        ns.append(n)
    assert len(set(ns)) >= 2, ns


def _run(args):
    r = subprocess.run([sys.executable] + args, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def test_entry_points_write_the_predicted_counts(cuda, tmp_path):
    from PIL import Image
    out = str(tmp_path)
    _run([os.path.join(ROOT, "code", "train.py"), "--count_head", "--nepochs", "1", "--batchsize", "2", "--synthetic", "2",
          "--output", os.path.join(out, "models")])
    ckpt = [f for f in os.listdir(os.path.join(out, "models", "CVPPP")) if f.endswith(".pth")][0]
    ckpt = os.path.join(out, "models", "CVPPP", ckpt)
    assert any(k.startswith("ins_cls_out.") for k in torch.load(ckpt, map_location="cpu"))
    gt_dir = os.path.join(out, "gt")
    os.makedirs(gt_dir)
    names, raws = [], []
    for j in range(2):
        nm = "plant%03d_rgb" % j
        raw = synth.leaf_image(j, 120, 110)
        Image.fromarray(raw).save(os.path.join(out, nm + ".png"))
        lab = synth.label_map(np.random.RandomState(j), 120, 110, 4).astype(np.int64) + 1
        lab[lab == 256] = 0
        Image.fromarray(lab.astype(np.uint8)).save(os.path.join(gt_dir, "plant%03d_label.png" % j))
        Image.fromarray((lab > 0).astype(np.uint8)).save(os.path.join(gt_dir, "plant%03d_fg.png" % j))
        names.append(os.path.join(out, nm + ".png"))
        raws.append(np.array(Image.open(names[-1]).convert('RGB')))
    with open(os.path.join(out, "val.lst"), "w") as f:
        f.write("\n".join(names) + "\n")
    with open(os.path.join(out, "counts.txt"), "w") as f:
        f.write("plant000,4\nplant001,4\n")
    _run([os.path.join(ROOT, "code", "pred_list.py"), "--count_head", "--lst", os.path.join(out, "val.lst"), "--model", ckpt,
          "--output", os.path.join(out, "pred")])
    sys.path.insert(0, os.path.join(ROOT, "code"))
    try:
        import _common
        model, pred = _common.build_model_and_prediction("CVPPP", ckpt, 0, count_head=True)
    finally:
        sys.path.pop(0)
    for j, raw in enumerate(raws):
        nm = "plant%03d_rgb" % j
        image, _, _ = pred.image_to_tensor(raw)
        want = int(model.predict_device_with_counts(image.unsqueeze(0))[2][0])
        got = np.load(os.path.join(out, "pred", nm, nm + "-n_objects.npy"))
        assert int(got) == want
    txt = _run([os.path.join(ROOT, "code", "evaluate.py"), "--pred_dir", os.path.join(out, "pred"), "--dataset", "CVPPP",
                "--names", os.path.join(out, "val.lst"), "--counts", os.path.join(out, "counts.txt"), "--gt_dir", gt_dir,
                "--empty_as_zero"])
    assert "MEAN |DIC|" in txt
