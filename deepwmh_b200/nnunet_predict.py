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
(upstream copies it; DeepWMH ignores it, predict.py:159-162).  Unless --disable_post_processing is given, a
`postprocessing.json` in the trainer folder is applied to each label file on the device and copied to the output folder,
as upstream's predict_cases does (DESIGN §11; DeepWMH passes the flag).  Any failure raises -> non-zero exit, which is what
`run_shell` turns into `exit(msg)` (deepwmh/utilities/external_call.py:63-72).  Flags of upstream nnUNet_predict that
DeepWMH never passes and this path does not implement are rejected loudly rather than ignored.

Besides DeepWMH's `-tr nnUNetTrainerV2`, the region-based BraTS trainer `-tr nnUNetTrainerV2BraTSRegions` is served
(DESIGN §12): sigmoid outputs, labels by its regions_class_order, trainer folder `nnUNetTrainerV2BraTSRegions__<plans>`.

Besides `-m 3d_fullres`, nnU-Net's cascade is served (DESIGN §13): `-m 3d_lowres` runs the plans' smallest stage from
`3d_lowres/<Task>/<tr>__<plans>`; `-m 3d_cascade_fullres` runs `3d_cascade_fullres/<Task>/<ctr>__<plans>` (-ctr, default
nnUNetTrainerV2CascadeFullRes) on the modalities plus the one-hot 3d_lowres labels, read from `-l <folder>/<case>.nii.gz`
or, without -l, predicted first with the -tr trainer into `<out>/3d_lowres_predictions` [U:predict_simple.py].
"""
from __future__ import annotations

import argparse
import os
import shutil
import sys
from typing import List

from . import cli as _cli
from . import postprocessing as _pp
from . import preprocess


def served_trainers():
    """-tr name -> trainer class.  Every other name (the BatchNorm BraTS variants among them) is refused."""
    from . import predictor
    return {"nnUNetTrainerV2": predictor.nnUNetTrainerV2, "nnUNetTrainerV2BraTSRegions": predictor.nnUNetTrainerV2BraTSRegions}


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


CONFIGS = (_cli.CONFIG, "3d_lowres", "3d_cascade_fullres")


def served_cascade_trainers():
    """-ctr name -> trainer class of the cascade's full-resolution stage."""
    from . import predictor
    return {"nnUNetTrainerV2CascadeFullRes": predictor.nnUNetTrainerV2CascadeFullRes}


def _model_folder(results: str, model: str, task: str, trainer: str):
    """<RESULTS_FOLDER>/nnUNet/<model>/<Task>/<trainer>__<plans> -> (folder, plans.pkl, checkpoint); a task id resolves to the
    task folder of that id."""
    cfg_dir = os.path.join(results, "nnUNet", model)
    if task.isdigit() and os.path.isdir(cfg_dir):               # upstream accepts a task id
        hits = [d for d in os.listdir(cfg_dir) if d.startswith("Task%03d_" % int(task))]
        if len(hits) != 1:
            raise RuntimeError("cannot resolve task id %s in %s" % (task, cfg_dir))
        task = hits[0]
    tdir = os.path.join(cfg_dir, task, "%s__%s" % (trainer, _cli.PLANNER))
    return tdir, os.path.join(tdir, "plans.pkl"), os.path.join(tdir, _cli.FOLD, "%s.model")


def _load_model(tdir: str, plans_path: str, ckpt_pattern: str, chk: str, model: str):
    """(plans, checkpoint path, stage) of a model folder; raises if a file is missing or a 3d_lowres folder's plans have no
    low-resolution stage."""
    ckpt_path = ckpt_pattern % chk
    for pth in (plans_path, ckpt_path):
        if not os.path.isfile(pth):
            raise RuntimeError('Cannot find "%s".' % pth)
    plans = _cli.load_plans(plans_path)
    stages = sorted(plans["plans_per_stage"].keys())
    if model == "3d_lowres":
        if len(stages) < 2:
            raise RuntimeError("%s has one plans stage, so it has no 3d_lowres stage (nnU-Net plans a low-resolution stage only "
                               "for large images)" % plans_path)
        return plans, ckpt_path, stages[0]
    return plans, ckpt_path, stages[-1]


def _pending(cases, output_folder: str, overwrite: bool, save_softmax: bool = False):
    todo = []
    for c in cases:
        out = os.path.join(output_folder, c + ".nii.gz")
        if overwrite or not os.path.isfile(out) or (save_softmax and not os.path.isfile(os.path.join(output_folder, c + "_0.nii.gz"))):
            todo.append(c)
    return todo


def _postprocessing(tdir: str, disabled: bool):
    """A model folder's postprocessing.json as (file, for_which_classes, min sizes), or Nones; a malformed file raises."""
    pp_file = os.path.join(tdir, "postprocessing.json")
    if disabled:
        return None, None, None
    if os.path.isfile(pp_file):
        return (pp_file,) + tuple(_pp.load_postprocessing(pp_file))
    print("WARNING! Cannot run postprocessing because the postprocessing file is missing. Make sure to run "
          "consolidate_folds in the output folder of the model first!\nThe folder you need to run this in is %s" % tdir)
    return None, None, None


def _predict_cases(trainer_class, plans, ckpt_path: str, stage: int, todo, inputs, output_folder: str, args, pp,
                   lowres_folder: str = None):
    import torch

    trainer = trainer_class(plans, device=0, max_batch=32 if not args.disable_tta else 16, stage=stage)   # CUDA_VISIBLE_DEVICES selects the GPU
    trainer.load_checkpoint_ram(torch.load(ckpt_path, map_location="cpu", weights_only=False), False)
    for c in todo:
        print("predicting", c)
        _cli.predict_case(trainer, plans, inputs[c], os.path.join(output_folder, c + ".nii.gz"),
                          softmax_file=os.path.join(output_folder, c + "_0.nii.gz") if args.save_softmax else None,
                          do_mirroring=not args.disable_tta, for_which_classes=pp[1], min_valid_object_sizes=pp[2],
                          segs_from_prev_stage=os.path.join(lowres_folder, c + ".nii.gz") if lowres_folder else None)
    trainer.network.close()


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(prog="nnUNet_predict", description="nnU-Net v1 inference on B200 (DeepWMH drop-in subset).")
    ap.add_argument("-i", "--input_folder", required=True, help="folder with <case>_0000.nii.gz (... <case>_000{M-1}.nii.gz) files")
    ap.add_argument("-o", "--output_folder", required=True)
    ap.add_argument("-t", "--task_name", required=True, help="task name or id, e.g. Task002_FinalModel")
    ap.add_argument("-tr", "--trainer_class_name", default="nnUNetTrainerV2",
                    help="trainer of 3d_fullres / 3d_lowres; with 3d_cascade_fullres, that of the 3d_lowres stage")
    ap.add_argument("-ctr", "--cascade_trainer_class_name", default="nnUNetTrainerV2CascadeFullRes",
                    help="trainer of the 3d_cascade_fullres stage")
    ap.add_argument("-m", "--model", default="3d_fullres", help="3d_fullres, 3d_lowres or 3d_cascade_fullres")
    ap.add_argument("-p", "--plans_identifier", default="nnUNetPlansv2.1")
    ap.add_argument("-f", "--folds", nargs="+", default=["all"])
    ap.add_argument("-chk", default="model_final_checkpoint", help="checkpoint name (DeepWMH: model_best / model_ep_XXXX)")
    ap.add_argument("-z", "--save_npz", action="store_true")
    ap.add_argument("--save_softmax", action="store_true", help="[fork] also write the background probability as <case>_0.nii.gz")
    ap.add_argument("--disable_tta", action="store_true", help="no mirroring (8x faster)")
    ap.add_argument("--disable_post_processing", action="store_true", help="do not apply the trainer folder's postprocessing.json (keep the largest component of its classes) to the label files")
    ap.add_argument("--selected_cases", nargs="+", default=None, help="[fork] only predict these case names")
    ap.add_argument("--overwrite_existing", action="store_true")
    ap.add_argument("--step_size", type=float, default=0.5)
    ap.add_argument("--num_parts", type=int, default=1)
    ap.add_argument("--part_id", type=int, default=0)
    ap.add_argument("--disable_mixed_precision", action="store_true")
    ap.add_argument("--all_in_gpu", default="None")
    ap.add_argument("--mode", default="normal")
    ap.add_argument("-l", "--lowres_segmentations", default="None",
                    help="3d_cascade_fullres: folder with the 3d_lowres labels <case>.nii.gz; without it 3d_lowres is predicted "
                         "first into <output_folder>/3d_lowres_predictions")
    ap.add_argument("--num_threads_preprocessing", type=int, default=6)
    ap.add_argument("--num_threads_nifti_save", type=int, default=2)
    args = ap.parse_args(argv)

    trainers = served_trainers()
    cascade_trainers = served_cascade_trainers()
    if args.trainer_class_name not in trainers or args.model not in CONFIGS or args.plans_identifier != _cli.PLANNER:
        raise NotImplementedError("this entry point serves -tr %s -m %s -p %s only (got -tr %s -m %s -p %s)"
                                  % (" | ".join(trainers), " | ".join(CONFIGS), _cli.PLANNER, args.trainer_class_name, args.model,
                                     args.plans_identifier))
    cascade = args.model == "3d_cascade_fullres"
    if cascade and args.cascade_trainer_class_name not in cascade_trainers:
        raise NotImplementedError("this entry point serves -ctr %s only (got -ctr %s)" % (" | ".join(cascade_trainers),
                                                                                         args.cascade_trainer_class_name))
    trainer_class = cascade_trainers[args.cascade_trainer_class_name] if cascade else trainers[args.trainer_class_name]
    if args.save_softmax and trainer_class.regions_class_order is not None:
        raise NotImplementedError("--save_softmax writes the background probability <case>_0.nii.gz; the region-based %s has no "
                                  "background output" % args.trainer_class_name)
    if list(args.folds) != [_cli.FOLD]:
        raise NotImplementedError("only `-f all` (DeepWMH trains one model on all data, predict.py:148)")
    if args.save_npz or args.mode != "normal" or args.disable_mixed_precision:
        raise NotImplementedError("-z / --mode / --disable_mixed_precision are not on DeepWMH's path")
    lowres_given = args.lowres_segmentations != "None"
    if lowres_given and not cascade:
        raise NotImplementedError("-l (the previous stage's segmentations) is the input of -m 3d_cascade_fullres only")
    if cascade and not lowres_given and (args.part_id != 0 or args.num_parts != 1):
        raise ValueError("without -l, 3d_cascade_fullres predicts 3d_lowres first, which needs --part_id 0 --num_parts 1 "
                         "(got --part_id %d --num_parts %d); predict 3d_lowres separately and pass its folder with -l"
                         % (args.part_id, args.num_parts))
    if args.all_in_gpu not in ("None", "False"):
        raise NotImplementedError("--all_in_gpu True (fp16 aggregation buffers) is not implemented; aggregation is fp32 on the device anyway")
    results = os.environ.get("RESULTS_FOLDER")
    if not results:
        raise RuntimeError("RESULTS_FOLDER is not set (DeepWMH sets it to the model directory, predict.py:101)")
    trainer_name = args.cascade_trainer_class_name if cascade else args.trainer_class_name
    tdir, plans_path, ckpt_pattern = _model_folder(results, args.model, args.task_name, trainer_name)
    plans, ckpt_path, stage = _load_model(tdir, plans_path, ckpt_pattern, args.chk, args.model)
    if cascade:
        trainer_class.input_channels(plans)                     # more inputs than the kernels take: refused here
        if not lowres_given:
            low = _model_folder(results, "3d_lowres", args.task_name, args.trainer_class_name)
            low_plans, low_ckpt, low_stage = _load_model(low[0], low[1], low[2], args.chk, "3d_lowres")
            low_pp = _postprocessing(low[0], False)             # upstream's low-resolution pass keeps its postprocessing

    cases = _cases_in(args.input_folder)
    if args.selected_cases is not None:
        missing = [c for c in args.selected_cases if c not in cases]
        if missing:
            raise RuntimeError("selected cases without an input file <case>_0000.nii.gz: %s" % ", ".join(missing))
        cases = [c for c in cases if c in set(args.selected_cases)]
    cases = cases[args.part_id::args.num_parts]                  # upstream's --part_id / --num_parts sharding
    n_mod = int(plans.get("num_modalities", 1))
    preprocess.normalization_schemes(plans)                      # an unknown scheme or missing CT constants: refused here
    inputs = {c: case_files(args.input_folder, c, n_mod) for c in cases}     # every modality present before any GPU work
    pp = _postprocessing(tdir, args.disable_post_processing)
    todo = _pending(cases, args.output_folder, args.overwrite_existing, args.save_softmax)
    lowres_folder = None
    if cascade:
        lowres_folder = args.lowres_segmentations if lowres_given else os.path.join(args.output_folder, "3d_lowres_predictions")
        if lowres_given:
            from . import nifti
            for c in todo:                                       # present, of the image's shape, labels of this model
                preprocess.read_prev_stage_labels(os.path.join(lowres_folder, c + ".nii.gz"), nifti.read_nifti(inputs[c][0])[1]["shape"],
                                                  int(plans["num_classes"]) + 1)
        else:
            preprocess.normalization_schemes(low_plans)
    os.makedirs(args.output_folder, exist_ok=True)
    shutil.copy(plans_path, args.output_folder)
    if pp[0] is not None:
        shutil.copy(pp[0], args.output_folder)
    print("number of cases:", len(cases), " number of cases that still need to be predicted:", len(todo))
    if not todo:
        return 0
    if args.step_size != 0.5:
        raise NotImplementedError("--step_size other than 0.5 is not passed by DeepWMH")

    if cascade and not lowres_given:
        print("lowres_segmentations is None. Attempting to predict 3d_lowres first...")
        os.makedirs(lowres_folder, exist_ok=True)
        shutil.copy(low[1], lowres_folder)
        if low_pp[0] is not None:
            shutil.copy(low_pp[0], lowres_folder)
        low_todo = _pending(todo, lowres_folder, args.overwrite_existing)
        low_args = argparse.Namespace(**dict(vars(args), save_softmax=False))
        _predict_cases(trainers[args.trainer_class_name], low_plans, low_ckpt, low_stage, low_todo, inputs, lowres_folder, low_args, low_pp)
        print("3d_lowres done")
    _predict_cases(trainer_class, plans, ckpt_path, stage, todo, inputs, args.output_folder, args, pp, lowres_folder)
    return 0


if __name__ == "__main__":
    sys.exit(main())
