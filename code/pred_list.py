"""pred_list.py -- a list of images -> one result directory per image, the file contract evaluate.py reads
(/root/reference/code/pred_list.py:14-22,54-99; the missing wae_opt argument of :54-57 is moot here).

    python code/pred_list.py --lst images.lst --model model.pth --output out_dir [--dataset CVPPP]
The list file holds one `image_path[,anything]` per line, as data/metadata/validation.lst does.
"""
import argparse
import os

import numpy as np

import _common

parser = argparse.ArgumentParser()
parser.add_argument('--lst', required=True, help='Text file that contains image paths')
parser.add_argument('--model', default='', help='Path of the model')
parser.add_argument('--usegpu', action='store_true', default=True)
parser.add_argument('--output', required=True, help='Path of the output directory')
parser.add_argument('--dataset', type=str, default='CVPPP')
parser.add_argument('--seed', type=int, default=0)
parser.add_argument('--count_head', action='store_true', help='Network with the instance-count head: each image is clustered '
                    'with its own predicted number of instances (the model must have been trained with --count_head)')

if __name__ == '__main__':
    opt = parser.parse_args()
    images_list = np.loadtxt(opt.lst, dtype='str', delimiter=',', ndmin=1)
    if images_list.ndim > 1:
        images_list = images_list[:, 0]
    image_names = [os.path.splitext(os.path.basename(p))[0] for p in images_list]
    model, prediction = _common.build_model_and_prediction(opt.dataset, opt.model, opt.seed, opt.count_head)
    from PIL import Image
    raws = (np.array(Image.open(str(p)).convert('RGB')) for p in images_list)
    kept = []

    def tee():                      # predict_many consumes the images in a worker thread; keep them for the writer
        for r in raws:
            kept.append(r)
            yield r

    written = 0
    for image_name, (fg_seg_pred, ins_seg_pred, n_objects_pred) in zip(image_names, prediction.predict_many(tee())):
        image = kept.pop(0)
        _common.write_prediction(os.path.join(opt.output, image_name), image_name, image, fg_seg_pred, ins_seg_pred, n_objects_pred)
        written += 1
    print('wrote %d of %d predictions under %s' % (written, len(image_names), opt.output))
