"""Which issue forms of conv3_tc_kernel the float64 layer checks reach (CPU: the host model in conv_paths.py).

Every case of test_gpu_layer_fp64 (CASES and BATCH_CASES) and of test_gpu_multimodal's layer cases is run through the model
with the B200's 148 SMs; the table of tags per case is printed, and the union must cover REQUIRED: every plane form and
launch form the kernel can reach.  Each tag of conv_paths.ALL_TAGS is either REQUIRED or named in UNREACHABLE with the
reason no network this library builds gets there; the claims that rest on the planner are checked by sweeping it below.
When a new issue form is added to the kernel (a new tag in conv_paths), it goes into REQUIRED and a case that reaches it
into test_gpu_layer_fp64.CASES -- this test names the tag until one does.
"""
import itertools

import pytest

import conv_paths as CP
from test_gpu_layer_fp64 import BATCH_CASES, CASES
from test_gpu_multimodal import LAYER_CASES, _layer_case_id, _plans as _mm_plans

NUM_SMS = 148

UNREACHABLE = {
    "KSTEPS=1": "build_plan requires feature counts that are multiples of 32, so KC0 >= 32, and tc_prepare finds a plan at "
                "kc = KC0 for every such layer (test_kc16_is_never_planned); the first conv has KC = 32",
    "general/nseg3": "a class spans at most 3 output planes and splits at most once at the ring wrap; with CB <= 128 (the "
                     "largest block tc_prepare picks) a segment holds >= 2 planes, and a transposed conv's class spans 1 "
                     "plane (test_general_path_needs_at_most_two_segments)",
}
REQUIRED = frozenset(t for t in CP.ALL_TAGS if t not in UNREACHABLE)

# the cases added to test_gpu_layer_fp64 (one or several, by name), and the tags only they reach.  At the production batch
# the 16^3 strided conv gets z-blocks longer than its ring of 4 slots: the only streamed-weight stride-(2,2,2) wrap.
ADDED_FOR = {
    ("dstride-32x64x64-n3",): {"dstride/nowrap", "dstride/wrap"},
    ("k133stream-4x64x64",): {"k133/stream"},
    ("nol32-72x80x40-n1-bf16",): {"bf16/XFORM/G=1"},
    ("bench-128^3-n32", "bench-128^3-n17-of-32"): {"s222/stream/wrap"},
}


def all_cases():
    """name -> (plans, batch size, activation type) of every float64 layer case on the tensor cores."""
    out = {}
    for name, (make, n, act, generic) in CASES.items():
        if not generic:
            out[name] = (make(), n, act)
    for name, (make, n, _max_batch, act, _samples) in BATCH_CASES.items():
        out[name] = (make(), n, act)
    for kind, M, C, base, act in LAYER_CASES:
        out["multimodal-" + _layer_case_id((kind, M, C, base, act))] = (_mm_plans(kind, M, C, base), 2, act)
    return out


def case_tags(cases):
    return {name: set().union(*(r["tags"] for r in CP.network_paths(p, n, act, NUM_SMS))) for name, (p, n, act) in cases.items()}


def missing(tags_by_case):
    covered = set().union(*tags_by_case.values())
    return sorted(REQUIRED - covered)


def test_required_and_unreachable_partition_the_vocabulary():
    assert set(UNREACHABLE) <= set(CP.ALL_TAGS), set(UNREACHABLE) - set(CP.ALL_TAGS)
    assert REQUIRED | set(UNREACHABLE) == set(CP.ALL_TAGS)


def test_fp64_cases_cover_every_reachable_issue_form():
    tags = case_tags(all_cases())
    for name, t in tags.items():
        print("%-32s %s" % (name, " ".join(sorted(t))))
    unknown = set().union(*tags.values()) - set(CP.ALL_TAGS)
    assert not unknown, ("tags outside the vocabulary (the model reached a form the kernel does not have)", unknown)
    reached_unreachable = set().union(*tags.values()) & set(UNREACHABLE)
    assert not reached_unreachable, reached_unreachable
    assert not missing(tags), ("issue forms no float64 layer case reaches", missing(tags))


@pytest.mark.parametrize("added", list(ADDED_FOR), ids=["+".join(a) for a in ADDED_FOR])
def test_added_cases_are_the_only_ones_reaching_their_forms(added):
    tags = case_tags(all_cases())
    for case in added:
        assert ADDED_FOR[added] <= tags[case], (case, ADDED_FOR[added] - tags[case])
    others = {k: v for k, v in tags.items() if k not in added}
    assert set(missing(others)) == ADDED_FOR[added], (added, missing(others))


# ------------------------------------------------------------------------------------------------
# the planner claims behind UNREACHABLE
# ------------------------------------------------------------------------------------------------
def _layer_shapes():
    """Every (c0, c1, cout, kernel, stride) build_plan can give a tcgen05 conv: features multiples of 32 up to 320, concat
    partners of equal width, stride only without a partner."""
    feats = range(32, 321, 32)
    strides = [s for s in itertools.product((1, 2), repeat=3)]
    for c0, cout, k, s in itertools.product(feats, feats, ((3, 3, 3), (1, 3, 3)), strides):
        if k[0] == 1 and s[0] != 1:
            continue
        yield c0, 0, cout, k, s
        if s == (1, 1, 1):
            yield c0, c0, cout, k, s


def test_kc16_is_never_planned():
    for c0, c1, cout, k, s in _layer_shapes():
        kp = CP.tc_prepare(c0, c1, cout, k, s, (32, 32, 32), tuple(32 // v for v in s))
        assert kp is not None and kp["KC"] >= 32, (c0, c1, cout, k, s, kp and kp["KC"])
        assert kp["CB"] <= 128
    for cin, cout, s in itertools.product(range(32, 321, 32), range(32, 321, 32), ((2, 2, 2), (1, 2, 2), (2, 1, 1))):
        kp = CP.tc_prepare_tconv(cin, cout, s, (8, 8, 8))
        assert kp is None or kp["KC"] >= 32, (cin, cout, s)


def test_general_path_needs_at_most_two_segments():
    # tc_prepare's blocks (CB <= 128, checked above) at both group counts: classes of 1-3 planes at every ring position;
    # transposed convs (CB up to 256): one plane
    for CB, G, cnt in itertools.product(range(16, 129, 16), (1, 2), (1, 2, 3)):
        R = min(CP.TC_MAX_R, (512 // G) // CB)
        for sl in range(R):
            assert CP.column_segments(sl, cnt, R, CB) <= 2, (CB, G, cnt, sl)
    for CB in range(32, 257, 32):
        R = 512 // CB
        assert all(CP.column_segments(sl, 1, R, CB) == 1 for sl in range(R))


# ------------------------------------------------------------------------------------------------
# known answers, worked by hand from the kernel
# ------------------------------------------------------------------------------------------------
def test_known_answer_128_dec4a_at_n32():
    """The benchmark's dec4-a (32 + 32 -> 32 channels on 128^3, layer 25) at the production batch: KC 32, CB 32, two
    resident-weight groups (R = 256 / 32 = 8), 128 tiles of 16 x 8, one z-block of all 128 planes (32 x 128 items fill
    148 SMs x 2 groups about 14 times; splitting D adds a 2-plane halo per block).  Inside the block the issuer starts at
    input plane -1, takes the general path at the block's first two planes, then stays in the steady state: lo_slot
    advances once per plane and passes every ring position, so all three wrap forms run; the last plane is general again."""
    from deepwmh_b200.plans import benchmark_plans
    rows = CP.network_paths(benchmark_plans(), 32, "fp16", NUM_SMS)
    r = rows[25]
    want = dict(kind="conv", KC=32, KSTEPS=2, CB=32, ncb=1, resident=1, SA=4, NB=18, R=8, G=2, ZB=128, nzb=1, tiles=128,
                items=32 * 128, grid=2048, xform=0, s222=0)
    assert {k: r["plan"][k] for k in want} == want
    assert r["kernel"] == "fp16<K2,SMALL_CB,DUAL>"
    assert r["tags"] == {"G=2", "KSTEPS=2", "SMALL_CB", "general/nseg1", "steady/res/nowrap", "steady/res/wrapA",
                         "steady/res/wrapB"}


def test_known_answer_no_wrap_on_a_two_plane_block():
    """On the 32^3 plan at n = 1 the 32-channel enc0-b (layer 1) is split into z-blocks of 2 planes (1 x 1 x 8 tiles
    would fill 3 % of the machine): output planes z, z + 1 take input planes z - 1 .. z + 2, three of which touch both
    outputs.  No plane has three live outputs, so the steady state never runs, and the ring (R = 8) never wraps: lo_slot
    reaches 1.  Every plane takes the general path with one segment."""
    from conftest import small_plans
    r = CP.network_paths(small_plans(), 1, "fp16", NUM_SMS)[1]
    assert (r["plan"]["ZB"], r["plan"]["nzb"], r["plan"]["R"], r["plan"]["tiles"]) == (2, 16, 8, 8)
    assert {t for t in r["tags"] if "/" in t and t.split("/")[0] in ("steady", "general", "s222", "dstride", "k133")} == \
        {"general/nseg1"}
