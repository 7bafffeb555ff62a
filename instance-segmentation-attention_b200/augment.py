"""Training on a directory of annotated images: the set is decoded once into device memory, and every batch is gathered
from there by one kernel that also applies the training-set augmentations (csrc/augment.cu, `isa_augment`).

    store = load_store('train.lst', gt_dir, ts.MAX_N_OBJECTS, ts.IMAGE_HEIGHT, ts.IMAGE_WIDTH, ts.MEAN, ts.STD, device)
    train = AugmentLoader(store, 16, ts, seed=ts.SEED, train=True)
    for images, sem, ins, n_objects in train: ...      # device tensors, the layouts Model.train_step reads

Input layout (CVPPP, as pred_list.py and evaluate.py read it): a list file with one image path per line (anything after
a comma is ignored); `<dir>/<base>_rgb.png` is the image and `<gt_dir>/<base>_label.png` its instance labels, a
palette or greyscale PNG whose pixel value is the instance id, 0 = background.

Geometry.  The reference's preprocessing code is not available, so what follows is this project's own specification
of the settings flags it names.  Every sample draws, from numpy.random.RandomState([seed, epoch]) after the epoch's
permutation and only for the flags that are on, in this order: a horizontal flip, a vertical flip, a transposition
(each with probability 1/2), k quarter turns counter-clockwise (k uniform in 0..3, as np.rot90) and a rotation by
theta ~ U[0, 360) degrees counter-clockwise about the centre.  With CENTER_CUT the rotated canvas keeps the extent
it had, so corners are cut (PIL rotate(expand=False)); without it the canvas grows to the smallest integer size that
holds the whole rotated image.  That canvas is then stretched to (IMAGE_HEIGHT, IMAGE_WIDTH).  With every flag off
this is the geometry of Prediction.image_to_tensor: the whole image stretched to the network size.  The inverse map
output -> source is composed in float64 and quantised to Q32.32 for the kernel.

Labels are sampled at the nearest source pixel and RGB bilinearly (zero outside the image), so a 530x500 -> 256x256
training view point-samples where PIL's resize in Prediction averages; see DESIGN.md section 4 for the difference.
"""
import ctypes
import math
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
from PIL import Image

from . import _lib, parallel

ONE = 1 << 32
COEF_LIMIT = 1 << 44        # |a_i| < 2^44, the kernel's bound (beyond it a sample is written empty)
MAX_SIDE = 32767

# settings flags that name augmentations this module does not implement
UNIMPLEMENTED = ("COLOR_JITTERING", "GRAYSCALING", "CHANNEL_SWAPPING", "GAMMA_ADJUSTMENT", "RESOLUTION_DEGRADING")
IMPLEMENTED = ("HORIZONTAL_FLIPPING", "VERTICAL_FLIPPING", "TRANSPOSING", "ROTATION_90X", "ROTATION", "CENTER_CUT")


def flags_from_settings(ts):
    """The geometry flags of a training-settings object -> dict; NotImplementedError for a flag that is on but names an
    augmentation this module does not apply."""
    for name in UNIMPLEMENTED:
        if getattr(ts, name, False):
            raise NotImplementedError("%s = True: this augmentation is not implemented" % name)
    return {name: bool(getattr(ts, name, False)) for name in IMPLEMENTED}


# ---------------------------------------------------------------------------------------------------- geometry
def inverse_map(h, w, H, W, hflip=False, vflip=False, transpose=False, k=0, theta=None, center_cut=False):
    """float64 (3,3) map from output pixel coordinates (pixel (x, y) spans [x, x+1) x [y, y+1)) to source coordinates,
    for a source of h x w pixels and an H x W output."""
    M = np.eye(3)
    cw, ch = float(w), float(h)

    def then(step):              # step: new canvas -> previous canvas
        nonlocal M
        M = M @ np.asarray(step, dtype=np.float64)

    if hflip:
        then([[-1, 0, cw], [0, 1, 0], [0, 0, 1]])
    if vflip:
        then([[1, 0, 0], [0, -1, ch], [0, 0, 1]])
    if transpose:
        then([[0, 1, 0], [1, 0, 0], [0, 0, 1]])
        cw, ch = ch, cw
    for _ in range(int(k) % 4):
        then([[0, -1, cw], [1, 0, 0], [0, 0, 1]])
        cw, ch = ch, cw
    if theta is not None:
        t = math.radians(float(theta))
        c, s = math.cos(t), math.sin(t)
        if center_cut:
            nw, nh = cw, ch
        else:                    # multiples of 90 degrees give exactly the swapped (or same) size
            nw = float(math.ceil(abs(c) * cw + abs(s) * ch - 1e-6))
            nh = float(math.ceil(abs(s) * cw + abs(c) * ch - 1e-6))
        then([[c, -s, cw / 2 - c * nw / 2 + s * nh / 2],
              [s, c, ch / 2 - s * nw / 2 - c * nh / 2],
              [0, 0, 1]])
        cw, ch = nw, nh
    then([[cw / W, 0, 0], [0, ch / H, 0], [0, 0, 1]])
    return M


def quantise(M):
    """(3,3) float64 map -> (a0..a5) int64 in Q32.32, the kernel's form."""
    a = np.round(np.asarray(M, dtype=np.float64)[:2, :].reshape(-1) * ONE)
    if not np.all(np.abs(a) < COEF_LIMIT):
        raise ValueError("map %s is outside the kernel's range (|entry| < 4096)" % np.asarray(M)[:2].tolist())
    return a.astype(np.int64)


def plain_map(h, w, H, W):
    """The un-augmented view (every flag off), exactly: a0 = round(w 2^32 / W), a4 = round(h 2^32 / H)."""
    return np.array([((w << 33) + W) // (2 * W), 0, 0, 0, ((h << 33) + H) // (2 * H), 0], dtype=np.int64)


def draw(rs, flags):
    """One sample's transform parameters, drawn from rs only for the flags that are on."""
    p = dict(hflip=False, vflip=False, transpose=False, k=0, theta=None, center_cut=flags.get("CENTER_CUT", False))
    if flags.get("HORIZONTAL_FLIPPING"):
        p["hflip"] = bool(rs.rand() < 0.5)
    if flags.get("VERTICAL_FLIPPING"):
        p["vflip"] = bool(rs.rand() < 0.5)
    if flags.get("TRANSPOSING"):
        p["transpose"] = bool(rs.rand() < 0.5)
    if flags.get("ROTATION_90X"):
        p["k"] = int(rs.randint(4))
    if flags.get("ROTATION"):
        p["theta"] = float(rs.uniform(0.0, 360.0))
    return p


def epoch_table(sizes, H, W, flags, seed, epoch):
    """-> (n, 7) int64 rows (source index, a0..a5): the epoch's permutation of the set and one drawn map per sample.
    sizes: [(h, w)] of the store's images.  The same (seed, epoch) gives the same table on every rank."""
    rs = np.random.RandomState([int(seed) & 0xffffffff, int(epoch) & 0xffffffff])
    perm = rs.permutation(len(sizes))
    table = np.empty((len(sizes), 7), dtype=np.int64)
    for i, src in enumerate(perm):
        h, w = sizes[src]
        table[i, 0] = src
        table[i, 1:] = quantise(inverse_map(h, w, H, W, **draw(rs, flags)))
    return table


def plain_table(sizes, H, W):
    """-> (n, 7) int64 rows (i, plain map of image i), in list order."""
    return np.array([[i] + list(plain_map(h, w, H, W)) for i, (h, w) in enumerate(sizes)], dtype=np.int64).reshape(-1, 7)


# ---------------------------------------------------------------------------------------------------- the kernel
def augment(store, params, H, W):
    """params: (b, 7) int64 device tensor -> (images (b,3,H,W) f32 channels_last, sem (b,H,W) u8, ins (b,H,W) u8,
    n_objects (b,) i32), all on the store's device and enqueued on its current stream."""
    lib = _lib.load()
    _lib.require_cuda(params, "params")
    params = params.contiguous()
    b = params.shape[0]
    dev = store.rgb.device
    image = torch.empty((b, H, W, 3), device=dev, dtype=torch.float32)
    sem = torch.empty((b, H, W), device=dev, dtype=torch.uint8)
    ins = torch.empty((b, H, W), device=dev, dtype=torch.uint8)
    nobj = torch.empty(b, device=dev, dtype=torch.int32)
    wsb = lib.isa_augment_workspace_bytes(b)
    ws = torch.empty(max(wsb, 4), device=dev, dtype=torch.uint8)
    rc = lib.isa_augment(store.rgb.data_ptr(), store.labels.data_ptr(), store.table.data_ptr(), store.n_images,
                         store.labels.numel(), params.data_ptr(), b, H, W, store.mean_std, image.data_ptr(),
                         sem.data_ptr(), ins.data_ptr(), nobj.data_ptr(), ws.data_ptr(), wsb, _lib.stream_ptr(dev))
    _lib.check(rc, "isa_augment")
    return image.permute(0, 3, 1, 2), sem, ins, nobj


# ---------------------------------------------------------------------------------------------------- the store
def read_list(path):
    """Image paths of a list file (pred_list.py --lst / evaluate.py --names format)."""
    names = np.loadtxt(path, dtype='str', delimiter=',', ndmin=1)
    if names.ndim > 1:
        names = names[:, 0]
    return [str(n) for n in names]


def label_path(image_path, gt_dir):
    base = os.path.splitext(os.path.basename(image_path))[0]
    if base.endswith('_rgb'):
        base = base[:-len('_rgb')]
    return os.path.join(gt_dir, base + '_label.png')


def read_pair(image_path, gt_dir, max_n_objects):
    """-> (rgb (h,w,3) u8, labels (h,w) u8 with ids 0..n-1 in ascending order of the PNG value, 255 = background).
    Raises ValueError naming the file for an input the store cannot hold."""
    lpath = label_path(image_path, gt_dir)
    with Image.open(image_path) as im:
        rgb = np.array(im.convert('RGB'))
    with Image.open(lpath) as im:
        if im.mode not in ('P', 'L'):
            raise ValueError("%s: label PNG of mode %s; expected P (palette) or L (greyscale)" % (lpath, im.mode))
        lab = np.array(im)
    if lab.shape != rgb.shape[:2]:
        raise ValueError("%s: label size %dx%d differs from the image's %dx%d (%s)"
                         % (lpath, lab.shape[1], lab.shape[0], rgb.shape[1], rgb.shape[0], image_path))
    if max(lab.shape) > MAX_SIDE:
        raise ValueError("%s: %dx%d is larger than %d pixels a side" % (image_path, lab.shape[1], lab.shape[0], MAX_SIDE))
    ids = np.unique(lab)
    ids = ids[ids != 0]
    if len(ids) == 0:
        raise ValueError("%s: no instance" % lpath)
    if len(ids) > max_n_objects:
        raise ValueError("%s: %d instances, more than MAX_N_OBJECTS = %d" % (lpath, len(ids), max_n_objects))
    lut = np.full(256, 255, dtype=np.uint8)
    lut[ids] = np.arange(len(ids), dtype=np.uint8)
    return rgb, lut[lab]


class ImageStore(object):
    """Decoded images packed in device memory: rgb [sum h*w*3] u8, labels [sum h*w] u8, table [n][3] i64 (pixel
    offset, h, w); `sizes` [(h, w)] and `names` stay on the host."""

    def __init__(self, names, rgbs, labels, mean, std, device):
        if len(names) == 0:
            raise ValueError("empty image list")
        self.names = list(names)
        self.sizes = [tuple(l.shape) for l in labels]
        self.n_images = len(self.names)
        offs = np.cumsum([0] + [h * w for h, w in self.sizes])
        table = np.array([[offs[i], h, w] for i, (h, w) in enumerate(self.sizes)], dtype=np.int64)
        dev = torch.device(device)
        self.rgb = torch.from_numpy(np.concatenate([r.reshape(-1) for r in rgbs])).to(dev)
        self.labels = torch.from_numpy(np.concatenate([l.reshape(-1) for l in labels])).to(dev)
        self.table = torch.from_numpy(table).to(dev)
        self.mean_std = (ctypes.c_float * 6)(*[float(v) for v in list(mean) + list(std)])

    @property
    def nbytes(self):
        return self.rgb.numel() + self.labels.numel() + self.table.numel() * 8


def load_store(list_path, gt_dir, max_n_objects, H, W, mean, std, device, workers=None):
    """Decodes every image of the list on a thread pool, compacts its ids, uploads the set once and checks that every
    image keeps an instance in its un-augmented H x W view (a sample whose augmented view loses every instance falls
    back to that view, so it must have one).  Raises ValueError naming the offending file."""
    if not 1 <= int(max_n_objects) <= 254:
        raise ValueError("MAX_N_OBJECTS = %d: ids are stored in a byte next to the background value 255" % max_n_objects)
    paths = read_list(list_path) if isinstance(list_path, str) else list(list_path)
    workers = workers or min(16, os.cpu_count() or 1)
    with ThreadPoolExecutor(max_workers=workers) as ex:     # PIL decodes with the GIL released
        pairs = list(ex.map(lambda p: read_pair(p, gt_dir, max_n_objects), paths))
    store = ImageStore(paths, [p[0] for p in pairs], [p[1] for p in pairs], mean, std, device)
    params = torch.from_numpy(plain_table(store.sizes, H, W)).to(store.rgb.device)
    counts = []
    for lo in range(0, store.n_images, 64):
        counts.append(augment(store, params[lo:lo + 64], H, W)[3].cpu())
    counts = torch.cat(counts).numpy()
    empty = [store.names[i] for i in np.nonzero(counts == 0)[0]]
    if empty:
        raise ValueError("%s: no instance left in the un-augmented %dx%d view (%d image(s) in all)"
                         % (label_path(empty[0], gt_dir), W, H, len(empty)))
    print("image store: %d images, %.1f MB on %s" % (store.n_images, store.nbytes / 1e6, store.rgb.device))
    return store


# ---------------------------------------------------------------------------------------------------- the loader
class AugmentLoader(object):
    """Yields (images, sem, ins, n_objects) device tensors from an ImageStore.

    train=True: each epoch draws a permutation and one map per image (epoch_table) and yields len // global_batch
    global batches, the last partial one dropped.  train=False: the un-augmented view in list order, every image once,
    the last batch partial.  Data parallel: every rank holds the whole store and computes the same global batches; it
    gathers only its parallel.shard_range slice of each.  A partial last validation batch smaller than the world is
    merged into the one before it, so no rank receives an empty batch."""

    def __init__(self, store, global_batch, H, W, flags=None, seed=0, train=True, rank=0, world=1):
        self.store, self.H, self.W = store, int(H), int(W)
        self.global_batch = int(global_batch)
        self.flags = dict(flags or {})
        self.seed, self.train = int(seed), bool(train)
        self.rank, self.world = int(rank), int(world)
        self.epoch = 0
        if self.global_batch < self.world:
            raise ValueError("global batch %d is smaller than the %d ranks" % (self.global_batch, self.world))
        n = store.n_images
        if train:
            if n < self.global_batch:
                raise ValueError("%d training images make no batch of %d" % (n, self.global_batch))
            self.bounds = [(j * self.global_batch, (j + 1) * self.global_batch) for j in range(n // self.global_batch)]
        else:
            if n < self.world:
                raise ValueError("%d validation images cannot be split over %d ranks" % (n, self.world))
            self.bounds = [(lo, min(lo + self.global_batch, n)) for lo in range(0, n, self.global_batch)]
            if len(self.bounds) > 1 and self.bounds[-1][1] - self.bounds[-1][0] < self.world:
                self.bounds[-2:] = [(self.bounds[-2][0], n)]
            self._plain = torch.from_numpy(plain_table(store.sizes, self.H, self.W)).to(store.rgb.device)

    def __len__(self):
        return len(self.bounds)

    def table(self, epoch):
        """The epoch's (n, 7) int64 parameter table on the device."""
        if not self.train:
            return self._plain
        t = torch.from_numpy(epoch_table(self.store.sizes, self.H, self.W, self.flags, self.seed, epoch))
        return t.pin_memory().to(self.store.rgb.device, non_blocking=True)

    def batches(self, epoch):
        params = self.table(epoch)
        for glo, ghi in self.bounds:
            lo, hi = parallel.shard_range(ghi - glo, self.rank, self.world)
            yield augment(self.store, params[glo + lo:glo + hi], self.H, self.W)

    def __iter__(self):
        epoch = self.epoch
        self.epoch += 1
        return self.batches(epoch)
