"""Shared by the entry points: import path + output writers of pred.py:59-92 / pred_list.py:67-99."""
import os
import sys

import numpy as np
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def spectral_colors(n):
    """Stand-in for plt.cm.Spectral (matplotlib is not installed): piecewise-linear 11-stop Spectral LUT."""
    stops = np.array([[158, 1, 66], [213, 62, 79], [244, 109, 67], [253, 174, 97], [254, 224, 139], [255, 255, 191],
                      [230, 245, 152], [171, 221, 164], [102, 194, 165], [50, 136, 189], [94, 79, 162]], dtype=np.float64)
    out = []
    for t in np.linspace(0, 1, max(n, 1)):
        x = t * (len(stops) - 1)
        i = min(int(x), len(stops) - 2)
        out.append(((1 - (x - i)) * stops[i] + (x - i) * stops[i + 1]).astype(np.uint8))
    return out


def write_prediction(out_dir, image_name, image, fg_seg_pred, ins_seg_pred, n_objects_pred):
    """<name>.png, -fg_mask.png (fg * 255), -ins_mask.png (uint8 labels), -ins_mask_color.png, -n_objects.npy"""
    os.makedirs(out_dir, exist_ok=True)
    n_clusters = len(np.unique(ins_seg_pred.flatten())) - 1
    colors = spectral_colors(n_clusters)
    color = np.zeros((ins_seg_pred.shape[0], ins_seg_pred.shape[1], 3), dtype=np.uint8)
    for i in range(n_clusters):
        color[ins_seg_pred == (i + 1)] = colors[i]
    Image.fromarray(image).save(os.path.join(out_dir, image_name + '.png'))
    Image.fromarray((fg_seg_pred * 255).astype(np.uint8)).save(os.path.join(out_dir, image_name + '-fg_mask.png'))
    Image.fromarray(ins_seg_pred).save(os.path.join(out_dir, image_name + '-ins_mask.png'))
    Image.fromarray(color).save(os.path.join(out_dir, image_name + '-ins_mask_color.png'))
    np.save(os.path.join(out_dir, image_name + '-n_objects.npy'), n_objects_pred)


def build_model_and_prediction(dataset, model_path, seed=0, count_head=False):
    """count_head: build the network with the instance-count head (the checkpoint must have been trained with it) and
    cluster each image with its predicted count."""
    from isa_b200.model import Model
    from isa_b200.prediction import Prediction
    from isa_b200 import settings
    ms = settings.CVPPPModelSettings() if dataset == 'CVPPP' else settings.CityscapesModelSettings()
    model = Model(dataset, ms.MODEL_NAME, ms.N_CLASSES, ms.MAX_N_OBJECTS,
                  use_instance_segmentation=ms.USE_INSTANCE_SEGMENTATION, use_coords=ms.USE_COORDINATES,
                  load_model_path=model_path or '', usegpu=True, n_embedding=ms.D_MODEL,
                  n_objects_prediction=ms.N_OBJECTS_PREDICTION, count_head=count_head or ms.COUNT_HEAD,
                  net_kwargs=dict(n_units=ms.N_RENET_UNITS, n_head=ms.N_HEAD, d_k=ms.D_K, d_v=ms.D_V))
    prediction = Prediction(ms.IMAGE_HEIGHT, ms.IMAGE_WIDTH, ms.MEAN, ms.STD, False, model, 1, seed=seed, strict=False)
    return model, prediction
