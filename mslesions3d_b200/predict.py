"""``predict.py`` entry point of the reference (``lesions3d/predict.py:29-44,235-323``) on the B200 path.

Same flags and the same ``predict_example(...)`` signature.  The reference reads NIfTI volumes through
MONAI/nibabel (absent here, and data loading is outside the accelerated path): this entry point accepts
a data-set directory in the generator's layout (``images/sub-XXXX_image.nii.gz`` + ``labels/sub-XXXX_seg.nii.gz``,
read by the package's own NIfTI-1 reader, ground-truth boxes extracted from the masks), a ``.npy``/``.pt`` stack
of volumes at ``--dataset_path`` or, by default, generates the synthetic cube volumes of
``generate_artificial_dataset.py`` in memory.  Checkpoints are the reference's
PyTorch-Lightning ``.ckpt`` files (``state_dict`` + ``hyper_parameters``).  Outputs follow the reference's
(predict.py:155-232,85-150,279-281): per subject ``sub-{id}_preds.csv`` / ``.json`` and the box-outline volume
``sub-{id}_preds.nii.gz`` (NIfTI-1 written by ``mslesions3d_b200/nifti.py``), ``aa_metrics_per_subject_(min_IoU=0.5|0.1).json`` from the device-side
``calculate_mAP``, plus one ``predictions.json`` with every subject's boxes / labels / scores.
With ``--window_overlap`` the volumes may be larger than the network input: they go through
``LSSD3D.predict_scans`` (sliding windows merged per scan) and every output refers to the whole scan.
"""
from __future__ import annotations

import argparse
import json
import os
from os.path import exists as pexists
from os.path import join as pjoin

import numpy as np
import torch

from . import synthetic
from .nifti import save_nifti
from .ssd3d import LSSD3D, device


def build_parser() -> argparse.ArgumentParser:
    parser = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    parser.add_argument('-d', '--dataset_path', type=str, default=r'../data/artificial_dataset',
                        help="data-set directory (images/*.nii.gz + labels/*.nii.gz) or a .npy/.pt stack of volumes "
                             "(N,C,D,H,W); synthetic volumes if it does not exist")
    parser.add_argument('-dn', '--dataset_name', type=str, help="name of dataset to use", default=None)
    parser.add_argument('-m', '--model_path', type=str, help="path to model", default=r'model_final.onnx')
    parser.add_argument('-mn', '--model_name', type=str, help="wandb model name", default=None)
    parser.add_argument('-p', '--percentage', type=float, help="percentage of the dataset to predict on", default=1.)
    parser.add_argument('-su', '--subject', type=str, default=None,
                        help="if prediction has to be done on 1 subject only, specify its id")
    parser.add_argument('-c', '--n_classes', type=int, help="number of classes in dataset", default=1)
    parser.add_argument('-nw', '--num_workers', type=int, default=8, help="number of workers for the dataset")
    parser.add_argument('-ps', '--predict_subset', type=str, help="subset to predict on",
                        choices=['train', 'validation', 'test', 'all'], default=r'train')
    parser.add_argument('-sc', '--min_score', type=float, default=0.5,
                        help="minimum score for a candidate box to be considered as positive")
    parser.add_argument('-k', '--top_k', type=int, default=100,
                        help="if there are a lot of resulting detection across all classes, keep only the top 'k'")
    parser.add_argument('-o', '--output_dir', type=str, help="path to output", default=r"../data/predictions/")
    parser.add_argument('-si', '--save_images', type=int, default=1,
                        help="whether to save the prediction volumes (NIfTI) and predictions.json")
    parser.add_argument('-bs', '--batch_size', type=int, default=8, help="volumes per forward (reference: 1)")
    parser.add_argument('-n', '--n_subjects', type=int, default=16, help="synthetic subjects when no dataset file")
    parser.add_argument('--window_overlap', type=float, default=None,
                        help="detect on whole scans larger than the network input: sliding input_size windows "
                             "overlapping by this fraction, merged per scan (LSSD3D.predict_scans)")
    parser.add_argument('--scan_size', type=int, nargs=3, default=None,
                        help="spatial size of the synthetic volumes (default: the model's input size)")
    return parser


def load_volumes(dataset_path, n_subjects, channels, size, percentage=1.0):
    if dataset_path and os.path.isfile(dataset_path):
        vols = np.load(dataset_path) if dataset_path.endswith(".npy") else torch.load(dataset_path).numpy()
        vols = vols.astype(np.float32)
    else:
        vols = synthetic.make_batch(n_subjects, channels, size)
    n = max(1, int(round(vols.shape[0] * percentage)))
    return vols[:n]


def box_outline_segmentation(det_boxes, det_labels, det_scores, img_shape, min_score):
    """The reference's prediction volume (predict.py:181-216): box j's outline is painted with the value j+1 into
    an array of the image's shape; boxes below ``min_score`` or with label 0 (the "nothing found" placeholder,
    ssd3d.py:437-440) are skipped.  -> (volume, scores_map [(label_id, score)], infos {label_id: (fractional box,
    voxel box, label, score)})."""
    seg = np.zeros(tuple(img_shape))
    scores_map, infos = [], {}
    shape2 = torch.tensor(list(img_shape) * 2, dtype=torch.float32)
    for j in range(det_boxes.shape[0]):
        score = float(det_scores[j])
        scores_map.append((j + 1, score))
        if score < min_score:
            continue
        label = int(det_labels[j])
        if label == 0:
            continue
        frac = [float(v) for v in det_boxes[j].tolist()]
        box = (torch.clip(det_boxes[j].float().cpu(), 0, 1) * shape2).numpy().astype(int).tolist()
        x0, y0, z0, x1, y1, z1 = box
        x0, y0, z0 = max(x0, 0), max(y0, 0), max(z0, 0)
        x1, y1, z1 = min(x1 + 1, img_shape[0] - 1), min(y1 + 1, img_shape[1] - 1), min(z1 + 1, img_shape[2] - 1)
        seg[x0, y0:y1, z0:z1] = j + 1
        seg[x1, y0:y1, z0:z1] = j + 1
        seg[x0:x1, y0, z0:z1] = j + 1
        seg[x0:x1, y1, z0:z1] = j + 1
        seg[x0:x1, y0:y1, z0] = j + 1
        seg[x0:x1, y0:y1, z1] = j + 1
        seg[x0:x1, y1, z1] = j + 1
        seg[x1, y0:y1, z1] = j + 1
        seg[x1, y1, z0:z1] = j + 1
        seg[x1, y1, z1] = j + 1
        infos[j + 1] = (frac, box, label, score)
    return seg, scores_map, infos


def save_predictions_example(subjects, img_shape, det_locs, det_labels, det_scores, min_score=0.5,
                             output_dir=r"./predictions", save_images=True, affine=None):
    """Per subject ``sub-{id}_preds.csv`` (label_id, score), ``sub-{id}_preds.json`` (the reference's ``all_infos``)
    and the box-outline volume ``sub-{id}_preds.nii.gz`` (predict.py:155-232; float64 voxels like the reference's
    ``np.zeros(img_shape)``, written by the package's NIfTI-1 writer since nibabel is absent)."""
    if not pexists(output_dir):
        os.makedirs(output_dir)
    for i, subj in enumerate(subjects):
        seg, scores_map, infos = box_outline_segmentation(det_locs[i].cpu(), det_labels[i].cpu(), det_scores[i].cpu(),
                                                          img_shape, min_score)
        if save_images:
            save_nifti(pjoin(output_dir, f"sub-{subj}_preds.nii.gz"), seg, affine)
        with open(pjoin(output_dir, f"sub-{subj}_preds.csv"), "w") as f:
            f.write(",label_id,score\n")
            for r, (lid, sc) in enumerate(scores_map):
                f.write("%d,%d,%r\n" % (r, lid, sc))
        with open(pjoin(output_dir, f"sub-{subj}_preds.json"), "w") as f:
            json.dump(infos, f)


def compute_subjects_mAP(model, subjects, det, gt_boxes, gt_labels, output_dir=r"./predictions", min_iou=0.5):
    """Per-subject detection metrics with the device-side ``calculate_mAP`` (predict.py:85-150), written to
    ``aa_metrics_per_subject_(min_IoU=...).json`` like the reference."""
    from .utils import calculate_mAP

    def convert(v):
        if torch.is_tensor(v):
            return v.cpu().item() if v.numel() == 1 else v.cpu().tolist()
        return v

    det_locs, det_labels, det_scores = det
    all_metrics = {}
    for i, subj in enumerate(subjects):
        gb = torch.as_tensor(gt_boxes[i]).to(device).reshape(-1, 6).float()
        gl = torch.as_tensor(gt_labels[i]).to(device).long()
        out = calculate_mAP([det_locs[i]], [det_labels[i]], [det_scores[i]], [gb], [gl],
                            [torch.zeros((gl.shape[0],), dtype=torch.bool, device=device)], min_overlap=min_iou,
                            return_detail=True)
        metrics = {}
        for key, value in out.items():
            if isinstance(value, dict):
                metrics[key] = {str(k): convert(v) for k, v in value.items()}
            else:
                metrics[key] = convert(value)
        all_metrics[str(subj)] = metrics
    with open(pjoin(output_dir, f"aa_metrics_per_subject_(min_IoU={min_iou}).json"), "w") as f:
        json.dump(all_metrics, f, indent=4)
    return all_metrics


def predict_example(model_path, output_dir, dataset_path, dataset_name, n_classes=1, subject=None, percentage=1.,
                    predict_subset="train", min_score=0.5, top_k=10, num_workers=8, save_images=True, model_name=None,
                    batch_size=8, n_subjects=16, model=None, window_overlap=None, scan_size=None):
    torch.manual_seed(970205)
    output_dir = output_dir if dataset_name is None else pjoin(output_dir, dataset_name)
    output_dir = output_dir if model_name is None else pjoin(output_dir, model_name)
    output_dir = pjoin(output_dir, f"{predict_subset}_set", f"min_score_{min_score}")
    if not pexists(output_dir):
        os.makedirs(output_dir)

    if model is None:
        model = LSSD3D.load_from_checkpoint(model_path, min_score=min_score)
    model = model.to(device).eval()
    model.top_k = top_k
    model.min_score = min_score

    gt_boxes = gt_labels = None
    subjects = None
    if dataset_path and os.path.isdir(pjoin(dataset_path, "images")):
        # the generator's on-disk layout (generate_artificial_dataset.py:54-111): NIfTI volumes + masks
        subjects, vols, gt_boxes, gt_labels = synthetic.load_dataset_dir(dataset_path, with_boxes=True)
        n = max(1, int(round(len(subjects) * percentage)))
        subjects, vols, gt_boxes, gt_labels = subjects[:n], vols[:n], gt_boxes[:n], gt_labels[:n]
    elif dataset_path and os.path.isfile(dataset_path):
        vols = load_volumes(dataset_path, n_subjects, model.input_channels, tuple(model.input_size), percentage)
    else:   # synthetic cube volumes come with their ground-truth boxes (generate_artificial_dataset.py)
        n = max(1, int(round(n_subjects * percentage)))
        size = tuple(scan_size) if scan_size is not None else tuple(model.input_size)
        vols, gt_boxes, gt_labels = synthetic.make_batch(n, model.input_channels, size, with_boxes=True)
    if subjects is None:
        subjects = list(range(vols.shape[0]))
    if subject is not None:
        k = subjects.index(subject) if subject in subjects else int(subject)
        vols, subjects = vols[k:k + 1], subjects[k:k + 1]
        if gt_boxes is not None:
            gt_boxes, gt_labels = gt_boxes[k:k + 1], gt_labels[k:k + 1]
    det_locs, det_labels, det_scores = [], [], []
    with torch.no_grad():
        if window_overlap is not None:      # whole scans: boxes come back as fractions of the scan's shape
            det_locs, det_labels, det_scores = model.predict_scans(torch.from_numpy(np.ascontiguousarray(vols)),
                                                                   overlap=window_overlap)
        else:
            batches = ({"img": torch.from_numpy(vols[s:s + batch_size]).pin_memory()}
                       for s in range(0, vols.shape[0], batch_size))
            for locs, labels, scores in model.predict_batches(batches):      # Trainer.predict of the reference
                det_locs += locs
                det_labels += labels
                det_scores += scores
    results = {str(subjects[i]): {"boxes": det_locs[i].cpu().tolist(), "labels": det_labels[i].cpu().tolist(),
                                  "scores": det_scores[i].cpu().tolist()} for i in range(len(det_locs))}
    if output_dir is not None:
        if save_images:
            with open(pjoin(output_dir, "predictions.json"), "w") as f:
                json.dump(results, f)
        save_predictions_example(subjects, tuple(vols.shape[2:]), det_locs, det_labels, det_scores, min_score,
                                 output_dir, bool(save_images))
        if gt_boxes is not None:
            for iou in (0.5, 0.1):    # predict.py:279-281
                compute_subjects_mAP(model, subjects, (det_locs, det_labels, det_scores), gt_boxes, gt_labels,
                                     output_dir=output_dir, min_iou=iou)
    return results


def main(argv=None):
    args = build_parser().parse_args(argv)
    subsets = ["train", "validation", "test"] if args.predict_subset == 'all' else [args.predict_subset]
    for psubset in subsets:
        predict_example(model_path=args.model_path, output_dir=args.output_dir, dataset_path=args.dataset_path,
                        dataset_name=args.dataset_name, n_classes=args.n_classes, subject=args.subject,
                        percentage=args.percentage, predict_subset=psubset, min_score=args.min_score,
                        top_k=args.top_k, num_workers=args.num_workers, save_images=args.save_images,
                        model_name=args.model_name, batch_size=args.batch_size, n_subjects=args.n_subjects,
                        window_overlap=args.window_overlap, scan_size=args.scan_size)


if __name__ == "__main__":
    main()
