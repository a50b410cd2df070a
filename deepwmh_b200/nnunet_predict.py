"""`nnUNet_predict`-shaped process entry (SURVEY.md section 8b, process / CLI level) backed by libdeepwmh_b200.so.

DeepWMH reaches the hot path by spawning `nnUNet_predict` with exactly these command lines:

    nnUNet_predict -i <dir> -o <dir> -tr nnUNetTrainerV2 -m 3d_fullres -p nnUNetPlansv2.1 -t <Task> -f all -chk model_best
                   --disable_post_processing --selected_cases a b ...            (deepwmh/main/predict.py:153-156)
    nnUNet_predict ... -chk model_ep_%04d --save_softmax --disable_tta           (deepwmh/pipeline/DCNN_multistage.py:331-344)
    nnUNet_predict ... -chk model_best                                           (DCNN_multistage.py:531-535)

with RESULTS_FOLDER / CUDA_VISIBLE_DEVICES in the environment (predict.py:101,150).  This module accepts those flags with
the same meaning: inputs `<in>/<case>_0000.nii.gz` (models with M modalities: `<case>_0000 ... <case>_000{M-1}.nii.gz`, the
modality order of the training data), outputs `<out>/<case>.nii.gz` (uint8 labels 0 .. C-1), `<out>/<case>_0.nii.gz`
(background probability, the fork's --save_softmax, read back at DCNN_multistage.py:359) and a copy of plans.pkl
(upstream copies it; DeepWMH ignores it, predict.py:159-162).  Any failure raises -> non-zero exit, which is what
`run_shell` turns into `exit(msg)` (deepwmh/utilities/external_call.py:63-72).  Flags of upstream nnUNet_predict that
DeepWMH never passes and this path does not implement are rejected loudly rather than ignored.
"""
from __future__ import annotations

import argparse
import os
import shutil
import sys
from typing import List

from . import cli as _cli


def _cases_in(folder: str) -> List[str]:
    return sorted({f[:-len("_0000.nii.gz")] for f in os.listdir(folder) if f.endswith("_0000.nii.gz")})


def case_files(folder: str, case: str, num_modalities: int) -> List[str]:
    """`<folder>/<case>_0000.nii.gz ... <case>_%04d.nii.gz` (modality order); raises if one of them is missing."""
    files = [os.path.join(folder, "%s_%04d.nii.gz" % (case, m)) for m in range(num_modalities)]
    missing = [os.path.basename(f) for f in files if not os.path.isfile(f)]
    if missing:
        raise RuntimeError("case %s lacks modality file(s) %s in %s (the model takes %d modalities: %s_0000 ... %s_%04d.nii.gz)"
                           % (case, ", ".join(missing), folder, num_modalities, case, case, num_modalities - 1))
    return files


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="nnUNet_predict", description="nnU-Net v1 inference on B200 (DeepWMH drop-in subset).")
    ap.add_argument("-i", "--input_folder", required=True, help="folder with <case>_0000.nii.gz (... <case>_000{M-1}.nii.gz) files")
    ap.add_argument("-o", "--output_folder", required=True)
    ap.add_argument("-t", "--task_name", required=True, help="task name or id, e.g. Task002_FinalModel")
    ap.add_argument("-tr", "--trainer_class_name", default="nnUNetTrainerV2")
    ap.add_argument("-m", "--model", default="3d_fullres")
    ap.add_argument("-p", "--plans_identifier", default="nnUNetPlansv2.1")
    ap.add_argument("-f", "--folds", nargs="+", default=["all"])
    ap.add_argument("-chk", default="model_final_checkpoint", help="checkpoint name (DeepWMH: model_best / model_ep_XXXX)")
    ap.add_argument("-z", "--save_npz", action="store_true")
    ap.add_argument("--save_softmax", action="store_true", help="[fork] also write the background probability as <case>_0.nii.gz")
    ap.add_argument("--disable_tta", action="store_true", help="no mirroring (8x faster)")
    ap.add_argument("--disable_post_processing", action="store_true", help="accepted; no postprocessing.json is ever applied here")
    ap.add_argument("--selected_cases", nargs="+", default=None, help="[fork] only predict these case names")
    ap.add_argument("--overwrite_existing", action="store_true")
    ap.add_argument("--step_size", type=float, default=0.5)
    ap.add_argument("--num_parts", type=int, default=1)
    ap.add_argument("--part_id", type=int, default=0)
    ap.add_argument("--disable_mixed_precision", action="store_true")
    ap.add_argument("--all_in_gpu", default="None")
    ap.add_argument("--mode", default="normal")
    ap.add_argument("-l", "--lowres_segmentations", default="None")
    ap.add_argument("--num_threads_preprocessing", type=int, default=6)
    ap.add_argument("--num_threads_nifti_save", type=int, default=2)
    args = ap.parse_args(argv)

    if args.trainer_class_name != _cli.TRAINER or args.model != _cli.CONFIG or args.plans_identifier != _cli.PLANNER:
        raise NotImplementedError("this entry point serves DeepWMH's model identity only: -tr %s -m %s -p %s" % (_cli.TRAINER, _cli.CONFIG, _cli.PLANNER))
    if list(args.folds) != [_cli.FOLD]:
        raise NotImplementedError("only `-f all` (DeepWMH trains one model on all data, predict.py:148)")
    if args.save_npz or args.lowres_segmentations != "None" or args.mode != "normal" or args.disable_mixed_precision:
        raise NotImplementedError("-z / -l / --mode / --disable_mixed_precision are not on DeepWMH's path")
    if args.all_in_gpu not in ("None", "False"):
        raise NotImplementedError("--all_in_gpu True (fp16 aggregation buffers) is not implemented; aggregation is fp32 on the device anyway")
    results = os.environ.get("RESULTS_FOLDER")
    if not results:
        raise RuntimeError("RESULTS_FOLDER is not set (DeepWMH sets it to the model directory, predict.py:101)")
    task = args.task_name
    cfg_dir = os.path.join(results, "nnUNet", _cli.CONFIG)
    if task.isdigit() and os.path.isdir(cfg_dir):               # upstream accepts a task id
        hits = [d for d in os.listdir(cfg_dir) if d.startswith("Task%03d_" % int(task))]
        if len(hits) != 1:
            raise RuntimeError("cannot resolve task id %s in %s" % (task, cfg_dir))
        task = hits[0]
    tdir = os.path.join(cfg_dir, task, "%s__%s" % (_cli.TRAINER, _cli.PLANNER))
    plans_path = os.path.join(tdir, "plans.pkl")
    ckpt_path = os.path.join(tdir, _cli.FOLD, args.chk + ".model")
    for pth in (plans_path, ckpt_path):
        if not os.path.isfile(pth):
            raise RuntimeError('Cannot find "%s".' % pth)

    cases = _cases_in(args.input_folder)
    if args.selected_cases is not None:
        missing = [c for c in args.selected_cases if c not in cases]
        if missing:
            raise RuntimeError("selected cases without an input file <case>_0000.nii.gz: %s" % ", ".join(missing))
        cases = [c for c in cases if c in set(args.selected_cases)]
    cases = cases[args.part_id::args.num_parts]                  # upstream's --part_id / --num_parts sharding
    plans = _cli.load_plans(plans_path)
    n_mod = int(plans.get("num_modalities", 1))
    inputs = {c: case_files(args.input_folder, c, n_mod) for c in cases}     # every modality present before any GPU work
    os.makedirs(args.output_folder, exist_ok=True)
    shutil.copy(plans_path, args.output_folder)
    todo = []
    for c in cases:
        out = os.path.join(args.output_folder, c + ".nii.gz")
        if args.overwrite_existing or not os.path.isfile(out) or (args.save_softmax and not os.path.isfile(os.path.join(args.output_folder, c + "_0.nii.gz"))):
            todo.append(c)
    print("number of cases:", len(cases), " number of cases that still need to be predicted:", len(todo))
    if not todo:
        return 0

    import torch

    import deepwmh_b200
    trainer = deepwmh_b200.nnUNetTrainerV2(plans, device=0, max_batch=32 if not args.disable_tta else 16)   # CUDA_VISIBLE_DEVICES selects the GPU
    trainer.load_checkpoint_ram(torch.load(ckpt_path, map_location="cpu", weights_only=False), False)
    if args.step_size != 0.5:
        raise NotImplementedError("--step_size other than 0.5 is not passed by DeepWMH")
    for c in todo:
        print("predicting", c)
        _cli.predict_case(trainer, plans, inputs[c], os.path.join(args.output_folder, c + ".nii.gz"),
                          softmax_file=os.path.join(args.output_folder, c + "_0.nii.gz") if args.save_softmax else None,
                          do_mirroring=not args.disable_tta)
    trainer.network.close()
    return 0


if __name__ == "__main__":
    sys.exit(main())
