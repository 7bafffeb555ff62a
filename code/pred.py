"""pred.py -- one image -> masks.  Command line of /root/reference/code/pred.py:12-22 (its hard-coded
/media/snowday paths and the unpack bug of :110-123 are gone).

    python code/pred.py --image img.png --model model.pth --output out_dir [--dataset CVPPP] [--seed 0]
"""
import argparse
import os

import _common

parser = argparse.ArgumentParser()
parser.add_argument('--image', required=True, help='Path of the image')
parser.add_argument('--model', default='', help='Path of the model (state_dict .pth); random init if omitted')
parser.add_argument('--usegpu', action='store_true', default=True, help='Kept for parity; the hot path is GPU only')
parser.add_argument('--output', required=True, help='Path of the output directory')
parser.add_argument('--dataset', type=str, default='CVPPP', help='"CVPPP" or "Cityscapes"')
parser.add_argument('--seed', type=int, default=0, help='k-means seed (the reference is unseeded)')
parser.add_argument('--count_head', action='store_true', help='Network with the instance-count head: each image is clustered '
                    'with its own predicted number of instances (the model must have been trained with --count_head)')

if __name__ == '__main__':
    opt = parser.parse_args()
    assert opt.dataset in ['CVPPP', 'Cityscapes']
    model, prediction = _common.build_model_and_prediction(opt.dataset, opt.model, opt.seed, opt.count_head)
    image, fg_seg_pred, ins_seg_pred, n_objects_pred = prediction.predict(opt.image)
    image_name = os.path.splitext(os.path.basename(opt.image))[0]
    _common.write_prediction(opt.output, image_name, image, fg_seg_pred, ins_seg_pred, n_objects_pred)
    print('wrote', os.path.join(opt.output, image_name + '-ins_mask.png'))
