"""CPU: every persistent launch of the bench forward (configs 2-4) has a GPU case in tests/test_gpu_persistent.py that
walks the same host plan past the CTAs' first tile."""

import pytest

from tests import persistent_plans as pp

EXEMPT = ()  # plan keys without a GPU case: none


@pytest.fixture(scope="module")
def production():
    return pp.production()


def test_case_ids_are_unique():
    ids = [c["id"] for c in pp.CASES]
    assert len(ids) == len(set(ids))


def test_every_production_plan_has_a_case_past_the_first_tile(production):
    by_key = {}
    for c in pp.CASES:
        by_key.setdefault(pp.case_plan(c)["key"], []).append(c)
    rows, missing = [], []
    for cfg, fn, entry, a, p in production:
        if p["key"] in EXEMPT:
            continue
        bar = min(4.0, p["per_cta"])
        ok = []
        for c in by_key.get(p["key"], []):
            q = pp.case_plan(c)
            walks = q.get("alt_walks", [q])  # mbconv_fused: whichever tile shape its probe picks
            if all(w["per_cta"] >= bar and (w["partial_wave"] or not p["partial_wave"])
                   and (w["tail"] == p["tail"] if "tail" in p else True)
                   and (w["tail_late"] or not any(w.get("tail", (0, 0)))) for w in walks):
                ok.append((c, q))
        rows.append(f"config {cfg} {fn:12s} {' '.join(x for x in p['key'] if x)}: {p['tiles']} tiles / {p['grid']} CTAs "
                    f"= {p['per_cta']:.2f} per CTA -> " + (f"{ok[0][0]['id']} ({ok[0][1]['per_cta']:.2f} per CTA)" if ok else "NONE"))
        if not ok:
            missing.append((cfg, fn, p["key"], {k: v for k, v in a.items() if isinstance(v, int) and v < 1 << 16}))
    print("\n".join(rows))
    assert not missing, missing


def test_cases_meet_the_walk_bar_on_their_own():
    for c in pp.CASES:
        q = pp.case_plan(c)
        assert q is not None, c["id"]
        if c["entry"] != "expand_sums":  # expand_sums runs at the production batch: its automatic split depends on it
            assert c["N"] >= 2 and q["per_cta"] >= 1, c["id"]
        if c["entry"].startswith("conv_tc") and q["per_cta"] > 1:
            assert q["second_epilogue"], c["id"]


def test_production_walks_reach_the_steady_state(production):
    """The census is worth having: the bench launches walk many tiles per CTA."""
    dominant = {e: max(p["per_cta"] for _, _, en, _, p in production if en == e) for e in ("stem_tc2", "mbconv_t",
                                                                                            "mbconv_fused")}
    assert dominant["stem_tc2"] > 200 and dominant["mbconv_t"] > 50 and dominant["mbconv_fused"] > 50
    assert {e for _, _, e, _, _ in production} == set(pp.ENTRIES)
