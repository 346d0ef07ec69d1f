"""No GPU: the fp64 coverage tables of tests/test_gpu_gemm_fp64.py reach every tcgen05 GEMM kernel instance the
dispatchers can launch, with every CTA serving >= 3 tiles, according to the host-only plan queries
(irfd_conv_gemm_plan, irfd_conv_wgrad_plan).  A heuristic change that moves a case to another instance, or a new
instance, fails here until a case reaches it."""
import pytest

from speak_hack_b200 import ops
from test_gpu_gemm_fp64 import (AFFINE, BNBWD, BNBWD_RES, CASES, MODE_NAMES, PLAIN, PROD_CONV_LAUNCHES,
                                 PROD_WGRAD_LAUNCHES, STATS, STYLE, WGRAD_CASES)

SMS = 148  # num_sms() without a device


def conv_instances():
    """(kernel, mode, BLOCK_N, cluster, per-warp epilogue) of every conv instance dispatch_block_n / dispatch_halo /
    dispatch_box can launch.  cluster: 1 single CTA, 2 CTA pair with multicast weights, 3 CTA pair with 2-SM MMAs (the
    per-warp PLAIN / STATS / BNBWD epilogues only).  STYLE, the halo and the boxed kernels have one epilogue each."""
    out = set()
    for mode in range(6):
        for bn in (64, 128, 256):
            for cl in (1, 2, 3):
                if (cl > 1 and bn == 64) or (cl == 3 and mode not in (PLAIN, STATS, BNBWD)):
                    continue
                for epi in ((0,) if mode == STYLE else (1,) if cl == 3 else (0, 1)):
                    out.add(("per-tap", mode, bn, cl, epi))
    for mode in (PLAIN, STATS, STYLE, AFFINE):
        for bn in (64, 128):
            out.add(("halo", mode, bn, 1, 0))
    for mode in (PLAIN, AFFINE):
        for bn in (64, 128, 256):
            out.add(("boxed", mode, bn, 1, 0))
    return out


def _conv_key(mode, plan):
    kind = "halo" if plan["halo"] else "boxed" if plan["boxed"] else "per-tap"
    epi = plan["warp_epi"] if kind == "per-tap" else 0
    return (kind, mode, plan["block_n"], plan["cluster"], epi)


def _name(key):
    kind, mode, bn, cl, epi = key
    return f"{kind} {MODE_NAMES[mode]} BLOCK_N={bn} cluster={cl} warp_epi={epi}"


def _conv_plans(monkeypatch):
    plans = []
    for c in CASES:
        with monkeypatch.context() as m:
            for k, v in c.env:
                m.setenv(k, v)
            plan = ops.conv_plan(*c.plan_args())
        assert plan is not None, f"{c.name}: the launch would refuse {c}"
        plans.append((c, plan))
    return plans


def test_plan_query_reads_the_environment(monkeypatch):
    args = (63, 32, 32, 64, 128, 3, STATS, 1, False, 128)
    for k in ("IRFD_GEMM_CLUSTER", "IRFD_GEMM_2SM", "IRFD_WARP_EPI", "IRFD_CONV_HALO"):
        monkeypatch.delenv(k, raising=False)
    assert ops.conv_plan(*args)["cluster"] == 1 and ops.conv_plan(*args)["warp_epi"] == 1
    monkeypatch.setenv("IRFD_GEMM_CLUSTER", "1")
    assert ops.conv_plan(*args)["cluster"] == 2
    monkeypatch.setenv("IRFD_GEMM_2SM", "1")
    assert ops.conv_plan(*args)["cluster"] == 3
    monkeypatch.setenv("IRFD_WARP_EPI", "0")
    assert ops.conv_plan(*args)["cluster"] == 2 and ops.conv_plan(*args)["warp_epi"] == 0
    halo = (1, 64, 256, 64, 64, 3, PLAIN, 1, False, 0)
    assert ops.conv_plan(*halo)["halo"] == 1
    monkeypatch.setenv("IRFD_CONV_HALO", "0")
    assert ops.conv_plan(*halo)["halo"] == 0
    assert ops.conv_plan(1, 7, 7, 64, 64, 3, STATS) is None  # box tiles serve PLAIN / AFFINE only
    assert ops.wgrad_plan(4, 16, 16, 64, 64, 5) is None


def test_conv_plan_matches_geometry():
    for c, plan in _conv_plans(pytest.MonkeyPatch()):
        n, h, w = c.plan_args()[:3]
        geo = ops.conv_geometry(n, h, w, c.k, c.wgroups) if not c.a_shared else None
        if geo is not None:
            assert geo[0] == plan["boxed"], c.name
            if plan["boxed"]:
                assert plan["m_tiles"] == geo[4] * geo[5] * geo[6], c.name
        if not plan["boxed"]:
            assert plan["m_tiles"] == (n * h * w + 127) // 128, c.name
        assert plan["n_tiles"] * plan["block_n"] == c.cout, c.name
        pair = 2 if plan["cluster"] > 1 else 1
        assert plan["grid"] == min(plan["units"], SMS // pair) * pair, c.name


def test_conv_cases_reach_every_instance(monkeypatch):
    reached, ragged = {}, set()
    even = []
    for c, plan in _conv_plans(monkeypatch):
        key = _conv_key(c.mode, plan)
        pair = 2 if plan["cluster"] > 1 else 1
        slots = plan["grid"] // pair
        rounds = plan["units"] // slots
        if c.sampled:  # production launch shapes run as the train step runs them
            continue
        assert rounds >= 3, f"{c.name} ({_name(key)}): {plan['units']} units on {slots} CTA slots, < 3 per CTA"
        reached.setdefault(key, []).append(c.name)
        if plan["units"] % slots:
            ragged.add(key)
        elif rounds % 2 == 0:
            even.append(c.name)
    missing = sorted(conv_instances() - set(reached))
    assert not missing, "no fp64 case reaches: " + "; ".join(_name(k) for k in missing)
    unknown = sorted(set(reached) - conv_instances())
    assert not unknown, "cases reach instances this test does not know: " + "; ".join(_name(k) for k in unknown)
    no_ragged = sorted(conv_instances() - ragged)
    assert not no_ragged, "no case with a ragged last round reaches: " + "; ".join(_name(k) for k in no_ragged)
    assert even, "no case runs an even number of full rounds"


def test_conv_cases_cover_operand_variants(monkeypatch):
    plans = _conv_plans(monkeypatch)
    for mode in (PLAIN, STATS, AFFINE, BNBWD, BNBWD_RES):
        assert {c.wgroups for c, _ in plans if c.mode == mode} >= {1, 3}, MODE_NAMES[mode]
    assert {c.mode for c, _ in plans if c.a_shared} >= {STATS, AFFINE}
    assert any(c.bias for c, _ in plans if c.mode == PLAIN and c.wgroups == 1)
    for kind in ("per-tap", "halo"):
        combos = {(c.relu, c.res) for c, p in plans if c.mode == AFFINE and _conv_key(c.mode, p)[0] == kind}
        assert combos >= {(r, s) for r in (0, 1, 2) for s in (False, True)}, (kind, combos)
    ragged_m = {c.mode for c, _ in plans if (c.n * c.h * c.w) % 128}
    assert ragged_m >= {PLAIN, STATS, AFFINE}
    halo_w = {c.w for c, p in plans if p["halo"]}
    assert 256 in halo_w and any(c.n % 2 for c, p in plans if p["halo"])
    boxed = {(c.h, c.w) for c, p in plans if p["boxed"]}
    assert boxed >= {(56, 56), (28, 28), (250, 250)}


WGRAD_GEMMS = {("halo", 64), ("per-tap", 64), ("per-tap", 128), ("per-tap", 256)}


def test_wgrad_cases_reach_every_instance(monkeypatch):
    """GEMM kernels and split-K reduce kernels are counted separately: the reduce reads fp32 partials whichever GEMM
    wrote them."""
    gemms, reduces = set(), set()
    ragged = set()
    for c in WGRAD_CASES:
        with monkeypatch.context() as m:
            for k, v in c.env:
                m.setenv(k, v)
            plan = ops.wgrad_plan(*c.plan_args())
        assert plan is not None, f"{c.name}: the launch would refuse {c}"
        kind = ("halo" if plan["halo"] else "per-tap", plan["block_n"])
        gemms.add(kind)
        reduces.add(plan["reduce"])
        if plan["splits"] > 1 and plan["num_kb"] % plan["kb_per_split"]:
            ragged.add(kind[0])
    assert not WGRAD_GEMMS - gemms, f"no fp64 case reaches the wgrad GEMM {sorted(WGRAD_GEMMS - gemms)}"
    missing = set(range(len(ops.WGRAD_REDUCE_KERNELS))) - reduces
    assert not missing, "no fp64 case reaches " + ", ".join(ops.WGRAD_REDUCE_KERNELS[r] for r in sorted(missing))
    assert ragged >= {"halo", "per-tap"}, f"a ragged last split only in {ragged}"
    assert any(c.groups == 3 for c in WGRAD_CASES) and any(c.x_shared for c in WGRAD_CASES)
    assert any(c.beta for c in WGRAD_CASES) and any(c.reduce_taps == 9 for c in WGRAD_CASES)
    stem = [c for c in WGRAD_CASES if c.reduce_cin == 147]
    assert stem and all(ops.wgrad_plan(*c.plan_args())["reduce"] >= 2 for c in stem)  # padded K tail: no transpose


DEFAULT_ENV = ("IRFD_GEMM_CLUSTER", "IRFD_GEMM_2SM", "IRFD_WARP_EPI", "IRFD_CONV_HALO", "IRFD_WGRAD_HALO")


def _wgrad_key(plan):
    return ("halo" if plan["halo"] else "per-tap", plan["block_n"], ops.WGRAD_REDUCE_KERNELS[plan["reduce"]])


def test_production_instances_have_sampled_cases(monkeypatch):
    """Every instance the train step and d_step launch (from their recorded launch shapes) has a production-size case
    at one of those shapes: conv by (kernel, mode, BLOCK_N, cluster, epilogue), wgrad by (GEMM, BLOCK_N, reduce)."""
    for k in DEFAULT_ENV:
        monkeypatch.delenv(k, raising=False)
    launched = {_conv_key(a[6], ops.conv_plan(*a)) for a in PROD_CONV_LAUNCHES}
    sampled = [c for c in CASES if c.sampled]
    for c in sampled:
        assert not c.env and tuple(c.plan_args()) in set(PROD_CONV_LAUNCHES), f"{c.name} is not a production launch"
    covered = {_conv_key(c.mode, ops.conv_plan(*c.plan_args())) for c in sampled}
    missing = sorted(launched - covered)
    assert not missing, "no production-size case reaches: " + "; ".join(_name(k) for k in missing)

    launched = {_wgrad_key(ops.wgrad_plan(*a)) for a in PROD_WGRAD_LAUNCHES}
    sampled = [c for c in WGRAD_CASES if c.sampled]
    for c in sampled:
        assert not c.env and tuple(c.plan_args()) in set(PROD_WGRAD_LAUNCHES), f"{c.name} is not a production launch"
    covered = {_wgrad_key(ops.wgrad_plan(*c.plan_args())) for c in sampled}
    assert not launched - covered, f"no production-size wgrad case reaches {sorted(launched - covered)}"
