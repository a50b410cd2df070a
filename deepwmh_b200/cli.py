"""`DeepWMH_predict`-compatible entry point (deepwmh/main/predict.py:50-199) with the nnUNet_predict subprocess
(:133-156) replaced by an in-process call into libdeepwmh_b200.so.

Same flags (-i -n -m -o -g --skip-bfc --custom-task-name), same output tree
(<out>/001_Preprocessed_Images/<case>_0000.nii.gz, <out>/002_Segmentations/{001_raw,002_postproc_3mm,003_postproc_fov}),
same fail-fast behaviour (any error -> non-zero exit); the 3 mm spark removal (predict.py:158-163) runs on the device.  Additive: --gpus a,b,... shards the cases over GPUs
(one worker process per GPU, no collective); --device-bfc runs N4 bias-field correction on the first of those GPUs
(deepwmh_b200.n4, same -s 2 and 50x50x50x50 schedule) instead of the ANTs binary.  By default, as in the reference,
N4 is the external ANTs program (use --skip-bfc, --device-bfc or have N4BiasFieldCorrection on PATH).  External, exactly as in
the reference: ROBEX FOV masking (skipped with a notice unless ROBEX_DIR is set) and GIF previews.
"""
from __future__ import annotations

import argparse
import os
import pickle
import shutil
import subprocess
import sys
from typing import Dict, List, Tuple

import numpy as np

from . import nifti, preprocess

TRAINER, CONFIG, PLANNER, FOLD, CHECKPOINT = "nnUNetTrainerV2", "3d_fullres", "nnUNetPlansv2.1", "all", "model_best"


def find_model(model_root: str, custom_task: str = None) -> Dict[str, str]:
    """Model directory layout of deepwmh/main/install_model.py:18-43 / predict.py:101-107,138-147."""
    model_root = os.path.abspath(model_root)
    if not os.path.isdir(model_root):
        raise RuntimeError('Directory not exist: "%s".' % model_root)
    if not os.path.isdir(os.path.join(model_root, "nnUNet")):
        raise RuntimeError('Invalid model directory. Cannot find directory "nnUNet" in folder "%s".' % model_root)
    cfg_dir = os.path.join(model_root, "nnUNet", CONFIG)
    tasks = sorted(d for d in os.listdir(cfg_dir) if os.path.isdir(os.path.join(cfg_dir, d))) if os.path.isdir(cfg_dir) else []
    if custom_task is not None:
        task = custom_task
    elif len(tasks) == 0:
        raise RuntimeError('Cannot find any task folder in "%s".' % cfg_dir)
    elif len(tasks) > 1:
        raise RuntimeError('Found multiple task folders in "%s".' % cfg_dir)
    else:
        task = tasks[0]
    tdir = os.path.join(cfg_dir, task, "%s__%s" % (TRAINER, PLANNER))
    paths = {"task": task, "plans": os.path.join(tdir, "plans.pkl"),
             "checkpoint": os.path.join(tdir, FOLD, CHECKPOINT + ".model")}
    for k in ("plans", "checkpoint"):
        if not os.path.isfile(paths[k]):
            raise RuntimeError('Cannot find "%s".' % paths[k])
    return paths


def load_plans(path: str) -> Dict:
    with open(path, "rb") as f:
        return pickle.load(f)


def _check_cases(case_names: List[str], images: List[str]):
    if len(case_names) != len(images):
        raise RuntimeError("Number of input images (%d) should be equal to case names (%d)." % (len(images), len(case_names)))
    if len(set(case_names)) != len(case_names):
        print("case names contain duplicates.")
        sys.exit(1)
    ok = set("abcdefghijklmnopqrstuvwxyzABCDEFGHIJKLMNOPQRSTUVWXYZ0123456789_-")
    for c, p in zip(case_names, images):
        if not c or any(ch not in ok for ch in c):
            print('invalid case name "%s".' % c)
            sys.exit(1)
        if not os.path.isfile(p):
            print('cannot find image "%s".' % p)
            sys.exit(1)


def predict_case(trainer, plans: Dict, in_file, out_file: str, softmax_file: str = None, post3mm_file: str = None,
                 do_mirroring: bool = True, for_which_classes=None, min_valid_object_sizes=None):
    """One case the way nnUNet_predict's predict_cases does it (SURVEY.md A7/A10): preprocess_patient (crop -> transpose ->
    resample -> z-score), tiled prediction, transpose back, resample back, argmax, paste back, NIfTI.  in_file: the image, or
    the list of its modality files in channel order.  Everything between the file read and the file write stays on the device.
    for_which_classes / min_valid_object_sizes: a loaded postprocessing.json for the label file (postprocessing.py)."""
    files = [in_file] if isinstance(in_file, str) else list(in_file)
    data, _, props = trainer.preprocess_patient(files, as_numpy=False)
    _, softmax = trainer.predict_preprocessed_data_return_seg_and_softmax(
        data, do_mirroring=do_mirroring, mirror_axes=trainer.data_aug_params["mirror_axes"], use_sliding_window=True,
        step_size=0.5, use_gaussian=True, all_in_gpu=False, mixed_precision=True, return_device_tensors=True)
    tb = list(plans.get("transpose_backward", [0, 1, 2]))
    softmax = softmax.permute([0] + [i + 1 for i in tb])
    preprocess.save_segmentation_nifti_from_softmax(trainer.network, softmax, out_file, props, 1, None, softmax_file, post3mm_file,
                                                    for_which_classes, min_valid_object_sizes)


def robex_fov_masking(case_names: List[str], image_folder: str, post_3mm_folder: str, post_fov_folder: str, robex_dir: str):
    """deepwmh/main/predict.py:39-48,165-181: remove false positives outside the brain -- ROBEX (an external program,
    `$ROBEX_DIR/runROBEX.sh <flair> <brain_out> <mask_out>`) skull-strips the pre-processed FLAIR and the 3 mm-cleaned label map
    is multiplied with its mask: ((seg * mask) > 0.5) as float32 into 003_postproc_fov/<case>.nii.gz."""
    sh, binary = os.path.join(robex_dir, "runROBEX.sh"), os.path.join(robex_dir, "ROBEX")
    if not (os.path.isfile(sh) and os.path.isfile(binary)):
        raise RuntimeError("Cannot find 'runROBEX.sh' and 'ROBEX' binary file in folder '%s', be sure to download and install ROBEX "
                           "in your local machine and check the path given is correct." % robex_dir)
    for case in case_names:
        out_seg = os.path.join(post_fov_folder, case + ".nii.gz")
        if os.path.isfile(out_seg):
            try:
                nifti.read_nifti(out_seg)
                continue                                             # predict.py:41: skip what already loads
            except Exception:
                pass
        flair = os.path.join(image_folder, case + "_0000.nii.gz")
        brain_out = os.path.join(post_fov_folder, case + "_brain.nii.gz")
        brain_mask = os.path.join(post_fov_folder, case + "_mask.nii.gz")
        rc = subprocess.call([sh, flair, brain_out, brain_mask], stdout=subprocess.DEVNULL)
        if rc != 0:
            raise RuntimeError("runROBEX.sh failed with exit code %d for case %s" % (rc, case))
        dat, hdr = nifti.read_nifti(os.path.join(post_3mm_folder, case + ".nii.gz"))
        accept, _ = nifti.read_nifti(brain_mask)
        for f in (brain_out, brain_mask):
            if os.path.isfile(f):
                os.remove(f)
        nifti.write_nifti(out_seg, ((dat * accept) > 0.5).astype(np.float32), hdr, dtype=np.float32)


def _worker(gpu: int, cases: List[Tuple[str, str, str, str]], model: Dict[str, str]):
    import torch
    import deepwmh_b200
    plans = load_plans(model["plans"])
    trainer = deepwmh_b200.nnUNetTrainerV2(plans, device=gpu, max_batch=32)
    ckpt = torch.load(model["checkpoint"], map_location="cpu", weights_only=False)
    trainer.load_checkpoint_ram(ckpt, False)
    for case, src, dst, post in cases:
        predict_case(trainer, plans, src, dst, post3mm_file=post)
        print("predicted %s" % case)
    trainer.network.close()


def main(argv=None):
    ap = argparse.ArgumentParser(description="Do lesion segmentation using pre-trained/installed model (B200-native path).",
                                 formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    ap.add_argument("-i", "--input-images", type=str, nargs="+", required=True,
                    help="Input image paths for prediction. Multiple input image paths are supported.")
    ap.add_argument("-n", "--case-names", type=str, nargs="+", required=True, help="Case name for each input image.")
    ap.add_argument("-m", "--trained-model", type=str, required=True,
                    help="Root folder of the trained model (containing the entire directory structure).")
    ap.add_argument("-o", "--output-folder", type=str, required=True,
                    help="Folder where pre-processed input images and predicted segmentations will be stored.")
    ap.add_argument("-g", "--gpu", type=int, default=0, help="GPU id.")
    bfc = ap.add_mutually_exclusive_group()
    bfc.add_argument("--skip-bfc", action="store_true", help="[Advanced] Skip bias field correction.")
    bfc.add_argument("--device-bfc", action="store_true",
                     help="[B200] N4 bias-field correction on the GPU instead of the ANTs binary.")
    ap.add_argument("--custom-task-name", type=str, required=False, help="[Advanced] Find model in specified task to segment image.")
    ap.add_argument("--gpus", type=str, default=None, help="[B200] comma-separated GPU ids: shard the cases over several GPUs.")
    args = ap.parse_args(argv)

    images = [os.path.abspath(p) for p in args.input_images]
    _check_cases(args.case_names, images)
    os.environ["RESULTS_FOLDER"] = os.path.abspath(args.trained_model)
    model = find_model(args.trained_model, args.custom_task_name)
    n_mod = int(load_plans(model["plans"]).get("num_modalities", 1))
    if n_mod != 1:
        raise RuntimeError("the model in %s takes %d input modalities; DeepWMH_predict takes one image per case. Run "
                           "nnUNet_predict with <case>_0000 ... <case>_%04d.nii.gz input files instead." % (args.trained_model, n_mod, n_mod - 1))
    print("model file is valid.")

    out = os.path.abspath(args.output_folder)
    image_folder = os.path.join(out, "001_Preprocessed_Images")
    raw_seg = os.path.join(out, "002_Segmentations", "001_raw")
    post_3mm = os.path.join(out, "002_Segmentations", "002_postproc_3mm")
    post_fov = os.path.join(out, "002_Segmentations", "003_postproc_fov")
    for d in (image_folder, raw_seg, post_3mm, post_fov):
        os.makedirs(d, exist_ok=True)

    gpus = [int(g) for g in args.gpus.split(",")] if args.gpus else [args.gpu]
    print("Pre-processing test images for prediction.")
    for case, src in zip(args.case_names, images):
        dst = os.path.join(image_folder, "%s_0000.nii.gz" % case)
        if args.device_bfc:
            from .n4 import n4_bias_field_correction
            d, h = nifti.read_nifti(src)
            nifti.write_nifti(dst, n4_bias_field_correction(d, 2, (50, 50, 50, 50), device=gpus[0]), h, dtype=np.float32)
        elif args.skip_bfc:
            if src.endswith(".gz"):
                shutil.copyfile(src, dst)
            else:
                d, h = nifti.read_nifti(src)
                nifti.write_nifti(dst, d, h, dtype=np.float32)
        else:
            n4 = shutil.which("N4BiasFieldCorrection")
            if n4 is None:
                raise RuntimeError("N4BiasFieldCorrection (ANTs) is not on PATH; bias-field correction is an external "
                                   "program in DeepWMH (predict.py:117-126). Re-run with --skip-bfc.")
            rc = subprocess.call([n4, "-d", "3", "-i", src, "-o", dst, "-c", "[50x50x50x50,0.0]", "-s", "2"])
            if rc != 0:
                raise RuntimeError("N4BiasFieldCorrection failed with exit code %d" % rc)

    work = [(c, os.path.join(image_folder, "%s_0000.nii.gz" % c), os.path.join(raw_seg, "%s.nii.gz" % c),
             os.path.join(post_3mm, "%s.nii.gz" % c)) for c in args.case_names]
    if len(gpus) == 1:
        _worker(gpus[0], work, model)
    else:
        import torch.multiprocessing as mp
        from .parallel import shard_cohort
        ctx = mp.get_context("spawn")
        procs = []
        for r, g in enumerate(gpus):
            mine = [work[i] for i in shard_cohort(len(work), r, len(gpus))]
            if mine:
                p = ctx.Process(target=_worker, args=(g, mine, model))
                p.start()
                procs.append(p)
        for p in procs:
            p.join()
            if p.exitcode != 0:
                raise RuntimeError("prediction worker failed with exit code %s" % p.exitcode)

    for case, _, seg_path, post_path in work:                                  # predict.py:158-163 ran inside the workers
        if not (os.path.isfile(seg_path) and os.path.isfile(post_path)):
            raise RuntimeError('prediction of case "%s" did not produce its outputs.' % case)
    final = post_3mm
    if os.environ.get("ROBEX_DIR"):
        robex_fov_masking(args.case_names, image_folder, post_3mm, post_fov, os.environ["ROBEX_DIR"])
        final = post_fov
    else:
        print("** ROBEX_DIR is not set: the brain-mask step (predict.py:165-181, an external program) is skipped and "
              "003_postproc_fov stays empty; the 3 mm-cleaned label maps are the result.")
    print("")
    print(">>> Prediction done.")
    print('>>> Raw/preprocessed images can be found in folder "%s".' % image_folder)
    print('>>> Segmentation results can be found in folder "%s".' % final)
    print("")
    return 0


if __name__ == "__main__":
    sys.exit(main())
