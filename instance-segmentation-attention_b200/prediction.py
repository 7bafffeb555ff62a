"""`Prediction` with the reference's API (/root/reference/code/lib/prediction.py:10-124):

    Prediction(resize_height, resize_width, mean, std, use_coordinates, model, n_workers)
    .predict(image_path) -> (raw_image HxWx3, sem_seg uint8 HxW, ins_seg uint8 HxW (0 = bg, 1..k), n_objects)
    .cluster(sem_seg_prediction, ins_seg_prediction, n_objects_prediction)

The CPU hop of the reference (.cpu().numpy() -> np.stack gather -> sklearn KMeans -> python scatter loop
-> cv2.resize, prediction.py:57-85,105-108) is replaced by the device pipeline of clustering.py:
argmax + foreground compaction, k-means++/Lloyd for all 35 restarts in one kernel, label scatter and
nearest up-sampling; only the two final uint8 masks are copied back.  A model with the count head
(`Model(count_head=True)`) clusters each image with its own predicted count: that count is k, a host argument of the
k-means kernels, so its 4 bytes are read back before the clustering is enqueued.  New argument `seed` (the reference
never seeds KMeans, so its output is not reproducible; here the default is 0).
Input images: RGB -> bilinear resize -> ToTensor -> Normalize(mean, std) (3 channels; the reference's
21-channel colour-space expansion needs scikit-image, which is not installed, and is data
preparation, not hot path).
"""
import sys

import numpy as np
import torch
from PIL import Image

from . import clustering


class Prediction(object):

    def __init__(self, resize_height, resize_width, mean, std, use_coordinates, model, n_workers, seed=0,
                 n_init=35, max_iter=500, strict=True):
        if use_coordinates:
            raise NotImplementedError("use_coordinates=True is off in every shipped setting and not implemented")
        self.mean = np.asarray(mean, dtype=np.float32).reshape(3, 1, 1)
        self.std = np.asarray(std, dtype=np.float32).reshape(3, 1, 1)
        self.use_coordinates = use_coordinates
        self.resize_height = resize_height
        self.resize_width = resize_width
        self.model = model
        self.n_workers = n_workers   # kept for signature parity; the GPU path has no worker pool
        self.seed = seed
        self.n_init = n_init
        self.max_iter = max_iter
        # strict=True raises like scikit-learn / the reference when an image cannot be clustered (fewer foreground
        # pixels than clusters, non-finite embeddings); strict=False (the list-processing scripts) writes an
        # all-background instance mask for that image and goes on
        self.strict = strict

    # ---- image loading (prediction.py:32-45)
    def image_to_tensor(self, img):
        """PIL RGB image or HxWx3 uint8 array -> (normalised (3,h,w) float tensor, raw_h, raw_w)."""
        if not isinstance(img, Image.Image):
            img = Image.fromarray(np.asarray(img, dtype=np.uint8))
        image_width, image_height = img.size
        img = img.convert('RGB').resize((self.resize_width, self.resize_height), Image.BILINEAR)
        x = np.asarray(img, dtype=np.float32).transpose(2, 0, 1) / 255.0
        x = (x - self.mean) / self.std
        return torch.from_numpy(np.ascontiguousarray(x)), image_height, image_width

    def get_image(self, image_path):
        return self.image_to_tensor(Image.open(image_path))

    # ---- clustering (prediction.py:52-85), device resident
    def cluster_device(self, sem_seg_prediction, ins_seg_prediction, n_objects_prediction, out_h=None, out_w=None):
        return clustering.cluster_embeddings(sem_seg_prediction, ins_seg_prediction, int(n_objects_prediction),
                                             out_h, out_w, seed=self.seed, n_init=self.n_init, max_iter=self.max_iter)

    def cluster(self, sem_seg_prediction, ins_seg_prediction, n_objects_prediction):
        """Same contract as the reference: tensors in, (sem uint8 (h,w), instance mask uint8 (h,w), n) numpy out."""
        dev = self.model.device
        n = int(np.asarray(torch.as_tensor(n_objects_prediction).cpu()).reshape(-1)[0])
        cls_map, ins_small, _, _, res = self.cluster_device(sem_seg_prediction.to(dev), ins_seg_prediction.to(dev), n)
        res.check()
        return cls_map.cpu().numpy(), ins_small.cpu().numpy(), n

    def upsample_prediction(self, prediction, image_height, image_width):
        """prediction.py:47-50 for callers that hold numpy masks (the fused path up-samples on the device)."""
        import cv2
        return cv2.resize(prediction, (image_width, image_height), interpolation=cv2.INTER_NEAREST)

    # ---- predict (prediction.py:87-124)
    def predict_array(self, raw_image):
        """raw_image HxWx3 uint8 -> (sem_seg uint8 HxW, ins_seg uint8 HxW, n_objects); one device->host copy of the masks
        (and, with the count head, one of the 4-byte count before the clustering)."""
        image, image_height, image_width = self.image_to_tensor(raw_image)
        sem, emb, n_pred = self.model.predict_device_with_counts(image.unsqueeze(0).pin_memory())
        n = self.model.n_objects_prediction if n_pred is None else int(n_pred[0])
        _, _, ins_up, cls_up, res = self.cluster_device(sem[0], emb[0], n, image_height, image_width)
        both = torch.stack([cls_up, ins_up]).cpu()     # the only D2H copy (also the sync point)
        if self.strict:
            res.check()
        else:
            try:
                res.check()
            except ValueError as e:
                sys.stderr.write("warning: image not clustered (%s); writing an empty instance mask\n" % e)
                return both[0].numpy(), np.zeros_like(both[1].numpy()), 0
        return both[0].numpy(), both[1].numpy(), n

    def predict_many(self, raw_images, prefetch=2):
        """Pipelined `predict_array` over an iterable of HxWx3 uint8 images (what pred_list.py does with a list of
        paths): a worker thread resizes / normalises / pins image i+1 (PIL releases the GIL) while the device works on
        image i, and the masks of image i are copied back asynchronously while image i+1 is enqueued.  The network of
        image i+1 is enqueued before the clustering of image i, so that waiting for image i's predicted count (count head)
        never leaves the device idle, except on the first image.
        Yields (sem_seg uint8 HxW, ins_seg uint8 HxW, n_objects) in order; results are identical to predict_array."""
        import queue
        import threading
        dev = self.model.device
        q = queue.Queue(maxsize=max(1, int(prefetch)))

        failure = []

        def producer():
            try:
                for raw in raw_images:
                    image, h, w = self.image_to_tensor(raw)
                    q.put((image.unsqueeze(0).pin_memory(), h, w))
            except BaseException as e:      # re-raised in the consumer: a failed load must not truncate the run silently
                failure.append(e)
            finally:
                q.put(None)

        threading.Thread(target=producer, daemon=True).start()
        ring = {}          # (h, w) -> two pinned staging buffers used alternately (masks + the k-means info words)
        counts = [torch.empty(1, dtype=torch.int32).pin_memory() for _ in range(2)]   # predicted counts, alternately

        def finish(p):
            host, info, ev, n = p
            ev.synchronize()
            if int(info[0]) != 0:
                msg = ("n_samples=%d should be >= n_clusters." % int(info[2]) if int(info[0]) == 1
                       else "Input X contains NaN or infinity.")
                if self.strict:
                    raise ValueError(msg)
                sys.stderr.write("warning: image not clustered (%s); writing an empty instance mask\n" % msg)
                return host[0].numpy().copy(), np.zeros_like(host[1].numpy()), 0
            return host[0].numpy().copy(), host[1].numpy().copy(), n

        staged = None      # network enqueued, clustering not yet: (sem, emb, h, w, pinned count or None, its event)
        pending = None     # clustering enqueued, masks on their way to the host: (host, host_info, event, n)
        n_images = 0
        turn = 0
        while True:
            item = q.get()
            nxt = None
            if item is not None:
                image, h, w = item
                sem, emb, n_pred = self.model.predict_device_with_counts(image)
                host_n = ev_n = None
                if n_pred is not None:
                    host_n = counts[n_images & 1]
                    host_n.copy_(n_pred[:1], non_blocking=True)
                    ev_n = torch.cuda.Event()
                    ev_n.record(torch.cuda.current_stream(dev))
                n_images += 1
                nxt = (sem, emb, h, w, host_n, ev_n)
            cur = None
            if staged is not None:
                sem, emb, h, w, host_n, ev_n = staged
                if host_n is None:
                    n = self.model.n_objects_prediction
                else:
                    ev_n.synchronize()       # the device is already running the next image's network
                    n = int(host_n[0])
                _, _, ins_up, cls_up, res = self.cluster_device(sem[0], emb[0], n, h, w)
                bufs = ring.get((h, w))
                if bufs is None:
                    bufs = ring[(h, w)] = [(torch.empty(2, h, w, dtype=torch.uint8).pin_memory(),
                                            torch.empty(16, dtype=torch.int32).pin_memory()) for _ in range(2)]
                host, host_info = bufs[turn & 1]
                turn += 1
                host[0].copy_(cls_up, non_blocking=True)
                host[1].copy_(ins_up, non_blocking=True)
                host_info.copy_(res.info, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(torch.cuda.current_stream(dev))
                cur = (host, host_info, ev, n)
            staged = nxt
            if pending is not None:
                yield finish(pending)
            pending = cur
            if item is None:
                break
        if pending is not None:
            yield finish(pending)
        if failure:
            raise failure[0]

    def predict(self, image_path):
        raw_image = np.array(Image.open(image_path).convert('RGB'))
        if not self.model.use_instance_segmentation:
            image, h, w = self.image_to_tensor(raw_image)
            sem = self.model.predict(image.unsqueeze(0))[0][1].numpy()
            return raw_image, self.upsample_prediction(sem, h, w)
        sem_seg, ins_seg, n = self.predict_array(raw_image)
        return raw_image, sem_seg, ins_seg, n
