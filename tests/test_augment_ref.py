"""CPU: the augmentation geometry (isa_b200.augment) and its numpy restatement (oracle/augment_ref.py) -- lossless
transforms, quarter-turn rotations, bilinear upscaling against PIL, the parameter table, and the loader's refusals."""
import os

import numpy as np
import pytest
from PIL import Image

from isa_b200 import augment as A
from isa_b200 import settings, synth
from oracle import augment_ref as R


def _img(seed, h, w):
    rs = np.random.RandomState(seed)
    return rs.randint(0, 256, size=(h, w, 3)).astype(np.uint8), rs.randint(0, 7, size=(h, w)).astype(np.uint8)


def _view(rgb, lab, **kw):
    h, w = lab.shape
    H, W = kw.pop("out", (h, w))
    a = A.quantise(A.inverse_map(h, w, H, W, **kw))
    return R.sample(rgb, lab, a, H, W)


@pytest.mark.parametrize("h,w", [(7, 5), (6, 6), (1, 9), (8, 1)])
@pytest.mark.parametrize("op", ["none", "hflip", "vflip", "transpose", "k1", "k2", "k3"])
def test_lossless_transforms_bit_exact(h, w, op):
    rgb, lab = _img(1, h, w)
    kw = {"none": {}, "hflip": dict(hflip=True), "vflip": dict(vflip=True), "transpose": dict(transpose=True),
          "k1": dict(k=1), "k2": dict(k=2), "k3": dict(k=3)}[op]
    ref = {"none": lambda a: a, "hflip": np.fliplr, "vflip": np.flipud, "transpose": lambda a: np.swapaxes(a, 0, 1),
           "k1": lambda a: np.rot90(a, 1), "k2": lambda a: np.rot90(a, 2), "k3": lambda a: np.rot90(a, 3)}[op]
    out_h, out_w = ref(lab).shape
    val, out_lab = _view(rgb, lab, out=(out_h, out_w), **kw)
    assert np.array_equal(out_lab, ref(lab))
    assert np.array_equal(val, ref(rgb).astype(np.float64))      # weights are 0 or 1 at pixel centres


@pytest.mark.parametrize("h,w", [(7, 5), (6, 6), (1, 4)])
@pytest.mark.parametrize("deg,k", [(90, 1), (180, 2), (270, 3)])
def test_free_rotation_by_quarter_turns_is_rot90(h, w, deg, k):
    rgb, lab = _img(2, h, w)
    want = np.rot90(lab, k)
    a = A.quantise(A.inverse_map(h, w, want.shape[0], want.shape[1], theta=deg))
    assert np.array_equal(a, A.quantise(A.inverse_map(h, w, want.shape[0], want.shape[1], k=k)))
    val, out_lab = R.sample(rgb, lab, a, want.shape[0], want.shape[1])
    assert np.array_equal(out_lab, want)
    assert np.array_equal(val, np.rot90(rgb, k).astype(np.float64))
    if h == w:      # a square keeps its extent, so CENTER_CUT gives the same view
        a_cut = A.quantise(A.inverse_map(h, w, h, w, theta=deg, center_cut=True))
        assert np.array_equal(a_cut, a)


def test_expanded_canvas_holds_the_whole_rotation():
    # 45 degrees: the canvas grows to ceil((w + h) / sqrt 2) a side and the source's corners land inside it
    M = A.inverse_map(100, 60, 114, 114, theta=45)
    fwd = np.linalg.inv(M)
    corners = fwd @ np.array([[0, 60, 0, 60], [0, 0, 100, 100], [1, 1, 1, 1]], dtype=np.float64)
    assert corners[:2].min() >= -1e-9 and corners[0].max() <= 114 + 1e-9 and corners[1].max() <= 114 + 1e-9


def test_upscale_matches_pil_bilinear():
    rgb, _ = _img(3, 20, 17)
    H, W = 57, 44
    val, _ = R.sample(rgb, np.zeros((20, 17), np.uint8), A.plain_map(20, 17, H, W), H, W)
    pil = np.asarray(Image.fromarray(rgb).resize((W, H), Image.BILINEAR)).astype(np.float64)
    # PIL renormalises its taps at the border where this kernel reads zeros (the black fill of PIL's rotate): compare
    # the output pixels whose four taps all lie inside the source
    ys = ((np.arange(H) + 0.5) * 20 / H - 0.5)
    xs = ((np.arange(W) + 0.5) * 17 / W - 0.5)
    iy = (ys >= 0) & (ys <= 19)
    ix = (xs >= 0) & (xs <= 16)
    d = np.abs(val - pil)[iy][:, ix]
    assert d.max() <= 1.0, d.max()


def test_all_flags_off_is_the_plain_resize_map():
    flags = {k: False for k in A.IMPLEMENTED}
    sizes = [(530, 500), (7, 3), (1, 1), (1024, 2048)]
    for (h, w) in sizes:
        assert np.array_equal(A.quantise(A.inverse_map(h, w, 256, 256)), A.plain_map(h, w, 256, 256))
        assert np.array_equal(A.plain_map(h, w, 256, 256), R.plain_map(h, w, 256, 256))
    t = A.epoch_table(sizes, 256, 256, flags, 23, 0)
    for row in t:
        h, w = sizes[row[0]]
        assert np.array_equal(row[1:], A.plain_map(h, w, 256, 256))
    assert sorted(t[:, 0]) == list(range(len(sizes)))


def test_table_is_a_function_of_seed_and_epoch():
    flags = A.flags_from_settings(settings.CVPPPTrainingSettings())
    sizes = [(530, 500), (480, 510), (300, 300)] * 5
    t0 = A.epoch_table(sizes, 256, 256, flags, 23, 0)
    assert np.array_equal(t0, A.epoch_table(sizes, 256, 256, flags, 23, 0))
    assert not np.array_equal(t0, A.epoch_table(sizes, 256, 256, flags, 23, 1))
    assert not np.array_equal(t0, A.epoch_table(sizes, 256, 256, flags, 24, 0))


def test_flags():
    ts = settings.CVPPPTrainingSettings()
    f = A.flags_from_settings(ts)
    assert all(f[k] for k in A.IMPLEMENTED)
    ts.GAMMA_ADJUSTMENT = True
    with pytest.raises(NotImplementedError, match="GAMMA_ADJUSTMENT"):
        A.flags_from_settings(ts)
    c = A.flags_from_settings(settings.CityscapesTrainingSettings())
    assert c["HORIZONTAL_FLIPPING"] and not (c["VERTICAL_FLIPPING"] or c["TRANSPOSING"] or c["ROTATION_90X"] or c["ROTATION"])


def test_renumber_and_fallback_in_the_oracle():
    lab = np.full((8, 8), 255, np.uint8)
    lab[0, 0], lab[4:, 4:] = 0, 3           # id 0 is one pixel, id 3 a block
    rgb = np.zeros((8, 8, 3), np.uint8)
    # 2x downscale: the sample at (1, 1) of each 2x2 cell; id 0 at (0, 0) is dropped, id 3 becomes 0
    out = R.augment([rgb], [lab], [[0] + list(A.plain_map(8, 8, 4, 4))], 4, 4, [0, 0, 0], [1, 1, 1])
    assert out["n_objects"][0] == 1 and set(np.unique(out["ins"][0])) == {0, 255}
    # a map that leaves the source entirely falls back to the plain view
    far = A.quantise(np.array([[1, 0, 100], [0, 1, 100], [0, 0, 1]], dtype=np.float64))
    out = R.augment([rgb], [lab], [[0] + list(far)], 8, 8, [0, 0, 0], [1, 1, 1])
    assert out["n_objects"][0] == 2 and np.array_equal(out["ins"][0], R.renumber(lab)[0])


# ---------------------------------------------------------------------------------------------------- loader refusals
def _write(tmp_path, name, rgb, lab, mode=None):
    Image.fromarray(rgb).save(os.path.join(str(tmp_path), name + "_rgb.png"))
    im = Image.fromarray(lab)
    if mode:
        im = im.convert(mode)
    im.save(os.path.join(str(tmp_path), "gt", name + "_label.png"))
    return os.path.join(str(tmp_path), name + "_rgb.png")


def _cvppp_label(seed, h, w, n):
    lab = synth.label_map(np.random.RandomState(seed), h, w, n).astype(np.int64) + 1
    lab[lab == 256] = 0
    return lab.astype(np.uint8)


@pytest.fixture
def gt(tmp_path):
    os.makedirs(os.path.join(str(tmp_path), "gt"))
    return os.path.join(str(tmp_path), "gt")


def test_read_pair_compacts_ids(tmp_path, gt):
    lab = np.zeros((30, 20), np.uint8)
    lab[:5], lab[10:15], lab[20:] = 7, 3, 200
    p = _write(tmp_path, "plant000", synth.leaf_image(0, 30, 20), lab)
    rgb, out = A.read_pair(p, gt, 32)
    assert rgb.shape == (30, 20, 3)
    assert np.array_equal(out[:5], np.full((5, 20), 1)) and np.array_equal(out[10:15], np.zeros((5, 20)))
    assert (out[20:] == 2).all() and (out[5:10] == 255).all()
    # a palette PNG reads the same
    p = _write(tmp_path, "plant001", synth.leaf_image(0, 30, 20), lab, mode="P")
    assert np.array_equal(A.read_pair(p, gt, 32)[1], out)


@pytest.mark.parametrize("case", ["size", "mode", "too_many", "empty"])
def test_loader_refuses_bad_input(tmp_path, gt, case):
    rgb = synth.leaf_image(1, 40, 36)
    lab = _cvppp_label(1, 40, 36, 4)
    if case == "size":
        lab = _cvppp_label(1, 41, 36, 4)
    elif case == "too_many":
        lab = _cvppp_label(1, 40, 36, 9)
    elif case == "empty":
        lab = np.zeros_like(lab)
    good = _write(tmp_path, "plant000", rgb, _cvppp_label(0, 40, 36, 4))
    bad = _write(tmp_path, "plant001", rgb, lab, mode="RGB" if case == "mode" else None)
    lst = os.path.join(str(tmp_path), "train.lst")
    with open(lst, "w") as f:
        f.write(good + "\n" + bad + "\n")
    msg = {"size": "differs", "mode": "mode RGB", "too_many": "more than MAX_N_OBJECTS", "empty": "no instance"}[case]
    with pytest.raises(ValueError, match=msg) as e:
        A.load_store(lst, gt, 8, 32, 32, [0.5] * 3, [0.2] * 3, "cpu")
    assert "plant001_label.png" in str(e.value)


def test_list_and_label_paths(tmp_path):
    lst = os.path.join(str(tmp_path), "a.lst")
    with open(lst, "w") as f:
        f.write("/data/A1/plant001_rgb.png,3\n/data/A1/plant002_rgb.png,5\n")
    names = A.read_list(lst)
    assert names == ["/data/A1/plant001_rgb.png", "/data/A1/plant002_rgb.png"]
    assert A.label_path(names[0], "/gt") == "/gt/plant001_label.png"
