"""CPU tier: every case of the conv conformance suite (conv_cases.py) lands on the plan its comment claims, and the cases
together reach every MMA issuer specialisation and every compiled epilogue variant of the conv kernel.

The planner (ops.conv_plan_ex) is host code, so a planner change that moves a case onto another branch fails here,
before the GPU tier runs."""
import collections

import numpy as np
import pytest

import conv_cases as cc
from conv_cases import ALL_CASES


@pytest.mark.parametrize("case", ALL_CASES, ids=lambda c: c.id)
def test_case_lands_on_its_plan(case):
    from oai_analysis_2_b200 import ops
    plan = cc.plan_of(ops, case)
    got = {k: plan[k] for k in case.expect}
    assert got == case.expect, f"{case.name} ({case.why}): plan {plan}"
    iss = cc.issuer(case, plan)
    # a case whose comment names an issuer must take it
    for name in cc.ISSUERS:
        if case.why.startswith(name + ":") or case.why.startswith(name + ","):
            assert iss == name, f"{case.name}: {case.why}, but the plan takes {iss}"
    # and one that names an epilogue variant must compile to it
    if "epilogue " in case.why:
        v = int(case.why.split("epilogue ")[1].split()[0])
        assert cc.epi_variant(case) == v, f"{case.name}: {case.why}, but the launch takes variant {cc.epi_variant(case)}"
    assert case.ab == bool(case.name.startswith("ab_")), "A/B-flag cases are named ab_* (and only they)"


def test_cases_cover_every_issuer_and_epilogue_variant():
    from oai_analysis_2_b200 import ops
    issuers, variants = collections.Counter(), collections.Counter()
    for case in ALL_CASES:
        issuers[cc.issuer(case, cc.plan_of(ops, case))] += 1
        variants[cc.epi_variant(case)] += 1
    # the A/B flags get their own cases; every issuer must also be reached without them (fast<3,2,4> through a
    # 24-channel source)
    plain = collections.Counter(cc.issuer(c, cc.plan_of(ops, c)) for c in ALL_CASES if not c.ab)
    print("issuer hits:", dict(sorted(issuers.items())))
    print("epilogue variant hits:", dict(sorted(variants.items())))
    assert set(cc.ISSUERS) <= set(issuers), f"issuers never hit: {set(cc.ISSUERS) - set(issuers)}"
    assert set(cc.ISSUERS) <= set(plain), f"issuers hit only through A/B flags: {set(cc.ISSUERS) - set(plain)}"
    assert set(cc.EPI_VARIANTS) <= set(variants), f"epilogue variants never hit: {set(cc.EPI_VARIANTS) - set(variants)}"
    modes = {cc.plan_of(ops, c)["mode"] for c in ALL_CASES}
    assert modes == set(cc.MODE_NAMES)
    # term codes 1-7 in both formats; those that allow one source on one and two sources
    seen = {(c.terms, c.fmt, c.c1 > 0) for c in ALL_CASES}
    for terms in range(1, 8):
        for fmt in (0, 1):
            for two in ((True,) if terms in (4, 5, 6) else (False,) if terms == 7 else (False, True)):
                assert (terms, fmt, two) in seen, f"terms {terms}, format {fmt}, two sources {two} not covered"
    c0s = {c.c0 for c in ALL_CASES}
    assert {8, 16, 24, 40, 96, 32, 64, 128, 512} <= c0s
    assert {64, 128, 256} <= {c.c1 for c in ALL_CASES}
    assert {32, 64, 96, 128, 192, 256, 384, 512} <= {c.cout for c in ALL_CASES}
    assert {1, 3} <= {c.NT for c in ALL_CASES}
    assert {1, 5, 9, 18} <= {c.D for c in ALL_CASES}


def test_kh_shared_tile_width_follows_the_grid():
    """A kh-shared layer narrower than 32 columns plans (and packs) with the tile width its launch takes."""
    from oai_analysis_2_b200 import ops
    for W, H in ((16, 16), (8, 16), (32, 8)):
        plan = ops.conv_plan_ex(4, H, W, 64, 0, 64, 0, 1, cc.KH_SHARED)
        assert plan["mode"] == cc.KH_SHARED_MODE and plan["nblk"] == 3
        w = np.zeros((64, 64, 3, 3, 3), np.float32)
        packed = ops.pack_conv_weights_ex(w, 64, 0, 4, H, W, 0, 1, flags=cc.KH_SHARED, device=None)
        assert packed.size == plan["packed_16B"] * 16


def test_kh_shared_rejects_a_grid_smaller_than_one_tile():
    from oai_analysis_2_b200 import _lib, ops
    with pytest.raises(_lib.OaiError, match="kh-shared mode needs"):
        ops.conv_plan_ex(4, 8, 8, 64, 0, 64, 0, 1, cc.KH_SHARED)   # an 8-wide tile needs 16 rows


def test_two_source_layers_reject_a_partial_first_source():
    from oai_analysis_2_b200 import _lib, ops
    with pytest.raises(_lib.OaiError, match="64-channel multiples"):
        ops.conv_plan_ex(4, 8, 16, 96, 64, 64)


def test_seg_layer_mirror_matches_the_planner():
    """conv_cases.SEG_LAYERS mirrors seg_net.cu's kLayers: every production spec is accepted with the packed size the
    mirror records (a change of seg_net.cu's table or of the planner then fails here instead of going unnoticed)."""
    from oai_analysis_2_b200 import ops
    regions = ops.seg_needed_regions(cc.PROD_TILE, cc.PROD_OVERLAP)
    cases = cc.production_cases(ops.seg_layer_terms(1), 0, regions)
    assert [c.name.split("_")[1] for c in cases] == [L[0] for L in cc.SEG_LAYERS]
    for case, layer in zip(cases, cc.SEG_LAYERS):
        assert cc.plan_of(ops, case)["packed_16B"] == layer[-1], case.name
        if case.region is not None:
            _, d_cnt, _, h_cnt = case.region[:4]
            assert d_cnt >= 1 and h_cnt >= 1
    # the mixed plan's lo8 layers are the ones whose storage the replay gives an e4m3 plane
    assert [c.terms for c in cases][-2:] == [6, 7]
    assert {c.name for c in cases if c.out == "lo8"} == {"prod_ec1_t1_f0", "prod_dc2_t6_f0"}


def test_w_box_entry_rejects_bad_arguments_with_messages():
    """oai_conv3d_igemm_box checks its box and the layer's kh-shared flag before it touches the device."""
    from oai_analysis_2_b200 import _lib
    from oai_analysis_2_b200._lib import c_size

    def box(box6, flags=cc.KH_SHARED):
        b = np.asarray(box6, dtype=np.int32)
        _lib.check(_lib.lib.oai_conv3d_igemm_box(None, 64, None, 0, 0, None, 1, 3, 16, 64, None, c_size(0), None, 64, 1,
                                                 0, 1, None, 0, None, flags, _lib.ptr(b), None), "conv3d_igemm_box")

    with pytest.raises(_lib.OaiError, match="outside the 3x16x64 grid"):
        box((0, 3, 0, 16, 40, 32))        # w beyond W
    with pytest.raises(_lib.OaiError, match="outside the 3x16x64 grid"):
        box((2, 2, 0, 16, 0, 8))          # d beyond D
    with pytest.raises(_lib.OaiError, match="outside the 3x16x64 grid"):
        box((0, 3, 4, 0, 0, 8))           # empty h range
    with pytest.raises(_lib.OaiError, match="kh-shared"):
        box((0, 3, 0, 16, 0, 8), flags=0)


def test_region_rows_restate_the_whole_tile_rule():
    by = {c.name: c for c in cc.ALL_CASES}
    assert cc.region_rows(by["reg_dc4"]) == (6, 58)            # TH = 2: rows 6 and 57 join the region's 7..56
    assert cc.region_rows(by["reg_kh_shared"]) == (9, 16)      # tiles at 9 and min(13, 16 - 4) = 12
    assert cc.region_rows(by["reg_k2s2"]) == (0, 16)           # one 8-row input tile, doubled
