"""A host model of which hand-written issue form of conv3_tc_kernel runs, plane by plane, for a given network and batch.

conv3_tc_kernel (deepwmh_b200/csrc/conv_tcgen05.cuh) issues its MMAs through one of several hand-written forms per input
plane -- the stride-1 steady state (one copy per weight mode, three accumulator-ring wrap forms each), the 1x3x3 loop, the
stride-(2,2,2) straight line (resident / streamed x wrap / no wrap), the depth-strided steady state and the general path
with 1-3 column segments -- and which one runs is decided by the host planner (tc_prepare, tc_plan_zb, the pairing rule
of tc_grid) together with the plane loop of the MMA issuer.  This module restates both in Python, line by line, so that
the test suite can say which of those forms its float64 layer checks reach.  Every statement cites the line it mirrors
(conv_tcgen05.cuh unless another file is named).  tests/test_gpu_conv_paths.py compares the plan half of it with the
library's own dwmh_layer_plan on the device, so the restatement cannot drift from the code unnoticed.

Vocabulary (one tag per plane form, plus per-launch tags):

    steady/{res,stream}/{nowrap,wrapA,wrapB}   stride-1 3x3x3 steady state (:587); wrapA: slots R-2, R-1 | 0, wrapB: R-1 | 0, 1
    k133/{res,stream}                           1x3x3, stride 1 (:698)
    s222/{res,stream}/{nowrap,wrap}            stride-(2,2,2) straight line (:739)
    dstride/{nowrap,wrap}                       depth-strided steady state (:809)
    general/nseg{1,2,3}                         general path, by the number of column segments of a class (:865)
    KSTEPS={1,2,4}, G=1, G=2, G=2->1/res, G=2->1/stream, FIRST/idle-group, FIRST, TCONV, XFORM, XFORM/G=1, SMALL_CB,
    {fp16,bf16}/{FIRST,TCONV,XFORM,XFORM/G=1,stream}   launch-level: template instantiation, pairing, activation type
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional

# conv_tcgen05.cuh:42-47
TC_TH, TC_TW = 16, 8
TC_MAX_SA, TC_MAX_NB, TC_MAX_R = 4, 40, 16
TC_SMEM_MAX, TC_SMEM_RESERVED = 232448, 5120
RAW32_MAX_EDGE = 64            # api.cu:61
MAX_NUM_FEATURES = 320         # predictor.py: d.max_num_features

# every plane-form tag of the issuer and every launch-level tag; network_paths() reports a subset of these
PATH_TAGS = tuple(
    ["steady/%s/%s" % (w, f) for w in ("res", "stream") for f in ("nowrap", "wrapA", "wrapB")]
    + ["k133/res", "k133/stream"]
    + ["s222/%s/%s" % (w, f) for w in ("res", "stream") for f in ("nowrap", "wrap")]
    + ["dstride/nowrap", "dstride/wrap"]
    + ["general/nseg1", "general/nseg2", "general/nseg3"])
LAUNCH_TAGS = tuple(
    ["KSTEPS=1", "KSTEPS=2", "KSTEPS=4", "G=1", "G=2", "G=2->1/res", "G=2->1/stream", "FIRST", "FIRST/idle-group", "TCONV",
     "XFORM", "XFORM/G=1", "SMALL_CB"]
    + ["%s/%s" % (a, k) for a in ("fp16", "bf16") for k in ("FIRST", "TCONV", "XFORM", "XFORM/G=1", "stream")])
ALL_TAGS = PATH_TAGS + LAUNCH_TAGS


# ------------------------------------------------------------------------------------------------
# the network's layers (api.cu build_plan, :136-200) and the commit-time decisions (dwmh_commit_weights)
# ------------------------------------------------------------------------------------------------
@dataclass
class Layer:
    kind: str                  # "first", "conv", "tconv"
    c0: int
    c1: int
    cout: int
    k: tuple
    s: tuple
    in_sp: tuple
    out_sp: tuple
    in0: int
    in1: int
    has_norm: bool
    raw32: bool = False
    s2d_s: tuple = (1, 1, 1)
    fused_norm: bool = False
    kp: Optional[dict] = None  # tcgen05 plan (None: CUDA-core kernels)


def network_layers(plans: Dict) -> List[Layer]:
    st = plans["plans_per_stage"][max(plans["plans_per_stage"].keys())]
    pools = [tuple(int(v) for v in p) for p in st["pool_op_kernel_sizes"]]
    kers = [tuple(int(v) for v in k) for k in st["conv_kernel_sizes"]]
    np_ = len(pools)
    f = [int(plans["base_num_features"])]                                                  # api.cu:140
    for i in range(1, np_ + 1):
        f.append(min(int(round(f[-1] * 2.0)), MAX_NUM_FEATURES))                            # api.cu:141
    sp = [tuple(int(v) for v in st["patch_size"])]                                         # api.cu:143
    for i in range(1, np_ + 1):
        sp.append(tuple(sp[i - 1][a] // pools[i - 1][a] for a in range(3)))                # api.cu:144-150
    L: List[Layer] = []

    def add_conv(c0, c1, cout, k, s, isp, osp, in0, in1, first):                           # api.cu:157-165
        L.append(Layer("first" if first else "conv", c0, c1, cout, k, s or (1, 1, 1), isp, osp, in0, in1, True))
        return len(L) - 1

    cur, cin, skip = -1, int(plans["num_modalities"]), []
    for e in range(np_):                                                                    # api.cu:169-176
        cur = add_conv(cin, 0, f[e], kers[e], pools[e - 1] if e > 0 else None, sp[e - 1] if e > 0 else sp[0], sp[e], cur, -1, e == 0)
        cur = add_conv(f[e], 0, f[e], kers[e], None, sp[e], sp[e], cur, -1, False)
        skip.append(cur)
        cin = f[e]
    cur = add_conv(cin, 0, f[np_], kers[np_], pools[np_ - 1], sp[np_ - 1], sp[np_], cur, -1, False)   # api.cu:178
    cur = add_conv(f[np_], 0, f[np_], kers[np_], None, sp[np_], sp[np_], cur, -1, False)              # api.cu:180
    ccur = f[np_]
    for u in range(np_):                                                                    # api.cu:182-196
        e = np_ - 1 - u
        sc = f[e]
        pk = pools[np_ - 1 - u]
        L.append(Layer("tconv", ccur, 0, sc, pk, pk, sp[e + 1], sp[e], cur, -1, False))
        tu = len(L) - 1
        cur = add_conv(sc, sc, sc, kers[np_ - u], None, sp[e], sp[e], tu, skip[e], False)
        cur = add_conv(sc, 0, sc, kers[np_ - u], None, sp[e], sp[e], cur, -1, False)
        ccur = sc
    last_conv = cur                                                                         # api.cu:197
    for i, l in enumerate(L):                                                               # api.cu:369-370
        l.raw32 = l.kind == "conv" and l.has_norm and i != last_conv and max(l.out_sp) <= RAW32_MAX_EDGE
    for l in L:                                                                             # api.cu:396-401
        strided = l.s != (1, 1, 1)
        k_ok = (l.k[0] == 3 or (l.k[0] == 1 and l.s[0] == 1)) and l.k[1] == 3 and l.k[2] == 3
        if l.kind == "conv" and strided and k_ok and l.c0 % 16 == 0 and l.c1 == 0 and l.cout % 16 == 0:
            L[l.in0].s2d_s = l.s
    for l in L:                                                                             # api.cu:437-461
        if l.kind == "first":
            if l.k == (3, 3, 3) and l.c0 <= 4:
                l.kp = tc_prepare_first(l.cout, l.out_sp, l.c0)
        elif l.kind == "tconv":
            l.kp = tc_prepare_tconv(l.c0, l.cout, l.s, l.in_sp)
        else:
            l.kp = tc_prepare(l.c0, l.c1, l.cout, l.k, l.s, l.in_sp, l.out_sp)
    uses = [0] * len(L)                                                                     # api.cu:480-487
    for l in L:
        if l.in0 >= 0:
            uses[l.in0] += 1
        if l.in1 >= 0:
            uses[l.in1] += 1
    for l in L:
        if l.kind != "conv" or l.kp is None or not l.kp["xform_ok"] or l.in0 < 0:
            continue
        P = L[l.in0]
        if P.has_norm and not P.raw32 and uses[l.in0] == 1 and P.s2d_s == (1, 1, 1) and P.cout <= 64:
            P.fused_norm = True
    return L


# ------------------------------------------------------------------------------------------------
# tc_prepare (:1237-1394), tc_prepare_tconv (:1398-1460), tc_prepare_first (:1467-1524): the plan fields only
# ------------------------------------------------------------------------------------------------
def tc_prepare(c0, c1, cout, k, s, in_sp, out_sp) -> Optional[dict]:
    if k[0] not in (3, 1) or k[1] != 3 or k[2] != 3:                                      # :1243
        return None
    kd = k[0]
    if kd == 1 and s[0] != 1:                                                               # :1245
        return None
    strided = s != (1, 1, 1)
    if strided and c1 > 0:                                                                  # :1247
        return None
    if c0 % 16 or c1 % 16 or cout % 16:                                                     # :1248
        return None
    cin = c0 + c1
    sd, sh, sw = s
    nclass = sd * sh * sw                                                                   # :1255
    Jlo = -1 if (sd == 1 and kd == 3) else 0
    Jhi = 1 if kd == 3 else 0
    jmax = 1 if kd == 1 else (3 if sd == 1 else 2)
    cls, tile0 = [], 0
    for cd in range(sd):                                                                    # :1261-1282
        for ph in range(sh):
            for pw in range(sw):
                pd = 1 - cd if sd == 2 else 0
                if kd == 1:
                    jlo, jcnt = 0, 1
                elif sd == 1:
                    jlo, jcnt = -1, 3
                elif pd == 0:
                    jlo, jcnt = 0, 1
                else:
                    jlo, jcnt = 0, 2
                mask, ntap = 0, 0
                for dy in range(3):
                    for dx in range(3):
                        kh = dy if sh == 1 else ((1 if dy == 1 else -1) if ph == 0 else (0 if dy == 0 else 2 if dy == 1 else -1))
                        kw = dx if sw == 1 else ((1 if dx == 1 else -1) if pw == 0 else (0 if dx == 0 else 2 if dx == 1 else -1))
                        if kh < 0 or kw < 0:
                            continue
                        mask |= 1 << (dy * 3 + dx)
                        ntap += 1
                cls.append(dict(jlo=jlo, jcnt=jcnt, tapmask=mask, tile0=tile0))
                tile0 += ntap
    tiles_per_kc = tile0                                                                    # :1283
    s222 = sd == 2 and sh == 2 and sw == 2 and nclass == 8 and tile0 == 18                # :1285-1293
    for c in range(8 if s222 else 0):
        cd, ph, pw = c >> 2, (c >> 1) & 1, c & 1
        mask = 0
        for iy in range(2 if ph else 1):
            for ix in range(2 if pw else 1):
                mask |= 1 << ((iy if ph else 1) * 3 + (ix if pw else 1))
        d = cls[c]
        if d["tapmask"] != mask or d["tile0"] != cd * 9 + ((5 if pw else 3) if ph else (1 if pw else 0)) or d["jlo"] != 0 \
                or d["jcnt"] != (2 if cd == 0 else 1):
            s222 = False
    KC0 = 64                                                                                # :1295-1296
    while KC0 > 16 and (c0 % KC0 or c1 % KC0):
        KC0 >>= 1
    budget = TC_SMEM_MAX - TC_SMEM_RESERVED                                                 # :1297
    KC = CB = SA = NB = resident = 0
    G = 1
    kc = KC0
    while kc >= 16 and not CB:                                                              # :1300-1312 dual resident
        a_stage, ntile = kc * 360, (cin // kc) * tiles_per_kc
        if ntile <= TC_MAX_NB:
            for cbt in range(min(cout, 64), 31, -16):
                if cout % cbt:
                    continue
                btot = ntile * jmax * cbt * kc * 2
                if btot + 2 * 3 * a_stage <= budget:
                    KC, CB, resident, NB, G = kc, cbt, 1, ntile, 2
                    SA = min(TC_MAX_SA, (budget - btot) // (2 * a_stage))
                    break
        kc >>= 1
    kc = KC0
    while kc >= 32 and not CB:                                                              # :1314-1323 dual streamed
        a_stage = kc * 360
        for cbt in range(min(cout, 64), 31, -16):
            if cout % cbt or 256 // cbt < jmax + 1:
                continue
            nb = (budget - 2 * 3 * a_stage) // (jmax * cbt * kc * 2)
            if nb >= 3:
                KC, CB, resident, SA, NB, G = kc, cbt, 0, 3, min(nb, TC_MAX_NB), 2
                break
        kc >>= 1
    kc = KC0
    while kc >= 16 and not CB:                                                              # :1325-1347 single group
        a_stage, ntile = kc * 360, (cin // kc) * tiles_per_kc
        if ntile <= TC_MAX_NB:
            for cbt in range(min(cout, 128), 15, -16):
                if cout % cbt:
                    continue
                if cbt < 32 and cbt != cout:
                    break
                btot = ntile * jmax * cbt * kc * 2
                if btot + 2 * a_stage <= budget:
                    KC, CB, resident, NB = kc, cbt, 1, ntile
                    SA = min(TC_MAX_SA, (budget - btot) // a_stage)
                    break
        if not CB:
            for cbt in range(min(cout, 128), 15, -16):
                if cout % cbt:
                    continue
                nb = (budget - 3 * a_stage) // (jmax * cbt * kc * 2)
                if nb >= 3:
                    KC, CB, resident, SA, NB = kc, cbt, 0, 3, min(nb, TC_MAX_NB)
                    break
        kc >>= 1
    if not CB:                                                                              # :1348
        return None
    xform_ok = not strided and kd == 3 and resident and c1 == 0 and KC == 32 and cin in (32, 64) and CB <= 32 and SA >= 3   # :1355
    return dict(kind="conv", first=False, tconv=False, KC=KC, CB=CB, ncb=cout // CB, SA=SA, NB=NB, resident=resident, G=G,
                R=min(TC_MAX_R, (512 // G) // CB),                                          # :1356 (the prepare-time G)
                D=out_sp[0], tilesH=-(-out_sp[1] // TC_TH), tilesW=-(-out_sp[2] // TC_TW), Din=in_sp[0] // sd,
                nclass=nclass, Jlo=Jlo, Jhi=Jhi, cls=cls, tiles_per_kc=tiles_per_kc, s222=s222, xform_ok=xform_ok)


def tc_prepare_tconv(cin, cout, s, in_sp) -> Optional[dict]:
    if cin % 16 or cout % 16:                                                               # :1402
        return None
    nco = s[0] * s[1] * s[2]
    CBt = 256 // nco                                                                        # :1404-1406
    while CBt >= 16 and (cout % CBt or CBt % 16):
        CBt -= 16
    if CBt < 16:
        return None
    CB = nco * CBt                                                                          # :1412-1413
    if CB % 32:
        return None
    KC = 64                                                                                 # :1414-1415
    while KC > 16 and cin % KC:
        KC >>= 1
    budget = TC_SMEM_MAX - TC_SMEM_RESERVED
    a_stage, b_tile, nkc = KC * 360, CB * KC * 2, cin // KC                                 # :1417
    if nkc <= TC_MAX_NB and nkc * b_tile + 2 * a_stage <= budget:                          # :1419-1424
        resident, NB, SA = 1, nkc, min(TC_MAX_SA, (budget - nkc * b_tile) // a_stage)
    else:
        resident, SA, NB = 0, 3, min((budget - 3 * a_stage) // b_tile, TC_MAX_NB)
        if NB < 2:
            return None
    return dict(kind="tconv", first=False, tconv=True, KC=KC, CB=CB, ncb=cout // CBt, SA=SA, NB=NB, resident=resident, G=1,
                R=512 // CB, D=in_sp[0], tilesH=-(-in_sp[1] // TC_TH), tilesW=-(-in_sp[2] // TC_TW), Din=in_sp[0],
                nclass=1, Jlo=0, Jhi=0, cls=[dict(jlo=0, jcnt=1, tapmask=1 << 4, tile0=0)], tiles_per_kc=1, s222=False,
                xform_ok=False)                                                             # :1409-1429


def tc_prepare_first(cout, sp, nmod) -> Optional[dict]:
    if cout not in (16, 32) or not 1 <= nmod <= 4:                                          # :1471-1472
        return None
    return dict(kind="first", first=True, tconv=False, KC=32, CB=cout, ncb=1, SA=TC_MAX_SA, NB=1, resident=1, G=2,
                R=min(TC_MAX_R, 256 // cout), D=sp[0], tilesH=-(-sp[1] // TC_TH), tilesW=-(-sp[2] // TC_TW), Din=sp[0],
                nclass=1, Jlo=0, Jhi=0, cls=[dict(jlo=0, jcnt=1, tapmask=1 << 4, tile0=0)], tiles_per_kc=1, s222=False,
                xform_ok=False)                                                             # :1476-1482


# ------------------------------------------------------------------------------------------------
# launch geometry: tc_plan_zb (:1549-1572) and tc_grid (the pairing rule)
# ------------------------------------------------------------------------------------------------
def tc_plan_zb(kp, nb, num_sms):
    tiles = kp["tilesH"] * kp["tilesW"]
    D = kp["D"]
    if not kp["first"] and not kp["tconv"] and D >= 16:                                    # :1551
        halo = kp["Jhi"] - kp["Jlo"]
        best, best_cost = D, -1
        for nzb in range(1, D // 2 + 1):                                                    # :1558-1565
            ZB = -(-D // nzb)
            if -(-D // ZB) != nzb:
                continue
            items = nb * kp["ncb"] * tiles * nzb
            ctas = -(-items // kp["G"])
            waves = -(-ctas // num_sms)
            cost = waves * (ZB + halo)
            if best_cost < 0 or cost < best_cost:
                best_cost, best = cost, ZB
        return best
    ZB = D                                                                                  # :1569-1571
    while nb * kp["ncb"] * tiles * (-(-D // ZB)) < 2 * num_sms and ZB > 2:
        ZB = (ZB + 1) // 2
    return ZB


def tc_grid(kp, nb, num_sms):
    tiles = kp["tilesH"] * kp["tilesW"]
    ZB = tc_plan_zb(kp, nb, num_sms)
    nzb = -(-kp["D"] // ZB)
    items = nb * kp["ncb"] * nzb * tiles
    G = kp["G"]
    if not kp["first"] and G == 2 and ((nzb * tiles) % 2 != 0 if kp["resident"] else tiles % 2 != 0):
        G = 1
    return dict(ZB=ZB, nzb=nzb, tiles=tiles, G=G, items=items, grid=-(-items // G))


# ------------------------------------------------------------------------------------------------
# the MMA issuer's plane loop (:559-940), replayed for one work item [z_lo, z_end)
# ------------------------------------------------------------------------------------------------
def column_segments(sl, cnt, R, CB):
    """Segments of the general path's MMAs for a class of cnt output planes starting at ring slot sl: split at the ring
    wrap and at N = 256 columns (:873-885)."""
    nseg, i = 0, 0
    while i < cnt:
        slot = sl + i if sl + i < R else sl + i - R
        ln = min(cnt - i, R - slot, 256 // CB)
        nseg += 1
        i += ln
    return nseg


def issuer_tags(kp, z_lo, z_end):
    """The plane forms the issuer takes for a work item on output planes [z_lo, z_end) (the same for every sample, cout
    block and tile: the choice depends on the plane range and the plan only)."""
    tags = set()
    R, CB, Din, Jlo, Jhi = kp["R"], kp["CB"], kp["Din"], kp["Jlo"], kp["Jhi"]
    res = "res" if kp["resident"] else "stream"
    t_first, t_last_nominal = z_lo - Jhi, z_end - 1 - Jlo                                  # :567
    plain = kp["nclass"] == 1 and Jlo == -1 and Jhi == 1                                    # :569
    lo_slot, next_fresh, zo_lo_prev = 0, z_lo, z_lo                                         # :575-576
    t = t_first - 1
    while t < t_last_nominal:                                                               # :577
        t += 1
        if t < 0 or t >= Din:                                                               # :578
            continue
        zo_lo, zo_hi = max(t + Jlo, z_lo), min(t + Jhi, z_end - 1)                          # :579
        if zo_lo != zo_lo_prev:                                                             # :580
            lo_slot = 0 if lo_slot + 1 == R else lo_slot + 1
            zo_lo_prev = zo_lo
        fresh_from = next_fresh                                                             # :581
        next_fresh = max(next_fresh, zo_hi + 1)                                             # :582-586
        if plain and zo_hi - zo_lo == 2 and R >= 3 and 3 * CB <= 256 and fresh_from == zo_hi:   # :587
            while True:
                wrap, wrapA = lo_slot + 3 > R, lo_slot + 2 == R                             # :600
                tags.add("steady/%s/%s" % (res, "wrapA" if wrapA else "wrapB" if wrap else "nowrap"))
                if t + 2 > z_end - 1 or t + 1 >= Din:                                       # :686
                    break
                t += 1                                                                      # :687
                lo_slot = 0 if lo_slot + 1 == R else lo_slot + 1                            # :688
                zo_lo_prev = t - 1                                                          # :689
                next_fresh += 1                                                             # :690-692
            continue                                                                        # :696
        if kp["nclass"] == 1 and Jlo == 0 and Jhi == 0 and kp["tiles_per_kc"] == 9 and fresh_from == zo_hi:   # :698
            tags.add("k133/%s" % res)
            continue
        if kp["s222"] and zo_lo == t and zo_hi == t + 1 and fresh_from == zo_hi and 2 * CB <= 256:           # :739
            tags.add("s222/%s/%s" % (res, "wrap" if lo_slot + 1 == R else "nowrap"))      # :801-802
            continue
        if Jlo == 0 and zo_lo == t and zo_hi == t + 1 and fresh_from == zo_hi and 2 * CB <= 256:            # :809
            tags.add("dstride/%s" % ("wrap" if lo_slot + 1 == R else "nowrap"))           # :813
            continue
        for c in kp["cls"]:                                                                 # :867-885
            dlo, dhi = max(t + c["jlo"], z_lo), min(t + c["jlo"] + c["jcnt"] - 1, z_end - 1)
            if dlo > dhi:
                continue
            cnt = dhi - dlo + 1
            sl = lo_slot + (dlo - zo_lo)
            if sl >= R:
                sl -= R
            nseg = column_segments(sl, cnt, R, CB)
            # the kernel keeps three segments in scalars: a fourth would be issued into the third's columns
            tags.add("general/nseg%d" % nseg if nseg <= 3 else "general/nseg>3 (unsupported)")
    return tags


def network_paths(plans: Dict, nb: int, act: str = "fp16", num_sms: int = 148, force_generic: bool = False) -> List[dict]:
    """Per layer (execution order): {"plan": the dwmh_layer_plan fields, "tags": the tags its launch at batch nb reaches,
    "kernel": the conv3_tc_kernel instantiation}."""
    L = network_layers(plans)
    out = []
    for i, l in enumerate(L):
        plan = dict(kind="cuda-core", kd=l.k[0], sd=l.s[0], sh=l.s[1], sw=l.s[2], act=act)
        if l.kp is None or force_generic:
            out.append(dict(plan=plan, tags=set(), kernel="CUDA cores"))
            continue
        kp = l.kp
        g = tc_grid(kp, nb, num_sms)
        xform = l.kind == "conv" and L[l.in0].fused_norm and kp["xform_ok"]                 # api.cu:681, tc_launch
        ks = kp["KC"] // 16
        plan.update(kind=kp["kind"], KC=kp["KC"], KSTEPS=ks, CB=kp["CB"], ncb=kp["ncb"], resident=int(kp["resident"]),
                    SA=kp["SA"], NB=kp["NB"], R=kp["R"], G=g["G"], ZB=g["ZB"], nzb=g["nzb"], tiles=g["tiles"],
                    items=g["items"], grid=g["grid"], xform=int(xform), s222=int(kp["s222"]))
        small = kp["CB"] <= 32 and not kp["tconv"]                                          # tc_launch: small
        # the instantiation tc_launch picks: conv3_tc_kernel<T, KSTEPS, SMALL_CB, TCONV, DUAL, XFORM, FIRST>
        if kp["first"]:
            flags = ["K2", "SMALL_CB", "DUAL", "FIRST"]
        elif xform:
            flags = ["K2", "SMALL_CB"] + (["DUAL"] if g["G"] == 2 else []) + ["XFORM"]
        elif kp["tconv"]:
            flags = ["K%d" % ks, "TCONV"]
        else:
            flags = ["K%d" % ks] + (["SMALL_CB"] if small else []) + (["DUAL"] if g["G"] == 2 else [])
        kernel = "%s<%s>" % (act, ",".join(flags))
        tags = set()
        if kp["first"]:
            tags |= {"FIRST", "%s/FIRST" % act}
            if g["items"] % 2:
                tags.add("FIRST/idle-group")                                                # :163-165: the last CTA's group 1 idles
        else:
            tags.add("KSTEPS=%d" % (2 if xform else ks))
            tags.add("G=%d" % g["G"])
            if kp["G"] == 2 and g["G"] == 1:
                tags.add("G=2->1/%s" % ("res" if kp["resident"] else "stream"))
            if "SMALL_CB" in flags:
                tags.add("SMALL_CB")
            if kp["tconv"]:
                tags |= {"TCONV", "%s/TCONV" % act}
            if xform:
                tags |= {"XFORM", "%s/XFORM" % act}
                if g["G"] == 1:
                    tags |= {"XFORM/G=1", "%s/XFORM/G=1" % act}
            if not kp["resident"]:
                tags.add("%s/stream" % act)
            for zb in range(g["nzb"]):
                tags |= issuer_tags(kp, zb * g["ZB"], min(kp["D"], (zb + 1) * g["ZB"]))
        out.append(dict(plan=plan, tags=tags, kernel=kernel))
    return out
