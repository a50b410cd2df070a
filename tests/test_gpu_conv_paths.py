"""The host model of the conv planner (conv_paths.py) against the library's own plan (dwmh_layer_plan), on the device.

For every layer of every float64 layer case the plan the launch would use -- kind, strides, KC / KSTEPS, CB, ncb, resident
weights, SA, NB, R, the tile pipelines per CTA after the pairing rule, ZB, nzb, tiles, items, grid, norm-on-load, the
stride-(2,2,2) path -- must equal the model's at the device's SM count.  So the coverage test_conv_paths.py computes from
the model is the coverage of the library, and a planner change that moves a case off the form it was added for fails here.
"""
import pytest
import torch

import conv_paths as CP
import oracle as O
from test_conv_paths import ADDED_FOR, all_cases
from test_gpu_layer_fp64 import BATCH_CASES

CASES = all_cases()
MAX_BATCH = {name: max_batch for name, (_m, _n, max_batch, _a, _s) in BATCH_CASES.items()}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_layer_plans_match_the_model(case):
    import deepwmh_b200
    plans, n, act = CASES[case]
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    net = O.build_benchmark_network(0, plans)
    tr = deepwmh_b200.nnUNetTrainerV2(plans, device=0, act_dtype=act, max_batch=MAX_BATCH.get(case, n))
    tr.load_checkpoint_ram({"state_dict": net.state_dict()}, False)
    nw = tr.network
    try:
        rows = CP.network_paths(plans, n, act, num_sms)
        assert len(rows) == nw.num_layers()
        bad = []
        for i, row in enumerate(rows):
            got = nw.layer_plan(i, n)
            want = dict(row["plan"])
            if want["kind"] == "cuda-core":
                got = {k: got[k] for k in want}
            if got != want:
                bad.append((i, {k: (got.get(k), want.get(k)) for k in set(got) | set(want) if got.get(k) != want.get(k)}))
        assert not bad, (case, "device plan != model plan (device, model)", bad)
        for added, tags in ADDED_FOR.items():
            if case in added:
                reached = set().union(*(r["tags"] for r in rows))
                assert tags <= reached, (case, "no longer reaches", tags - reached)
    finally:
        nw.close()
