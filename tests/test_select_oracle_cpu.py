"""The exact selection oracle without a GPU: its checkers flag every kind of wrong output, the override
emulation follows the kernel's summation order, every case of the exact plan matrix reaches the planner
branch it is meant to pin, and no test sets a CCR_* lever except through the helper that makes it take
effect."""
import ast
import os

import numpy as np
import pytest
import torch

import select_oracle as SO
from select_oracle import lever  # noqa: F401  (fixture)
from test_gpu_select_exact import CASES, case_mask, mask_args, plan_of, variants

TESTS = os.path.dirname(os.path.abspath(__file__))
K = 10


def _bf16(a):
    return torch.as_tensor(a, dtype=torch.float32).to(torch.bfloat16).float().numpy()


@pytest.fixture(scope="module")
def world():
    """Stored rows, a SET mask and the exact output for them: row 0 has an exact tie at rank 0 (a duplicated
    item), row 2 its best item masked, row 1 a +0.0 and a -0.0 in its top k."""
    rs = np.random.RandomState(5)
    R, N, D = 4, 200, 64
    q, items = _bf16(rs.standard_normal((R, D))), _bf16(rs.standard_normal((N, D)))
    x = q.astype(np.float64) @ items.astype(np.float64).T
    items[N - 1] = items[int(np.argmax(x[0]))]
    x = q.astype(np.float64) @ items.astype(np.float64).T
    top2 = int(np.argmax(x[2]))
    mask = (np.array([0, 0, 0, 1, 1]), np.array([top2], np.int32), np.array([-1e6]), SO.MASK_SET)
    vals = torch.as_tensor(x.astype(np.float32))
    vals[2, top2] = -1e6
    zeros = vals.clone()
    zeros[1] = -torch.arange(1, N + 1, dtype=torch.float32)
    zeros[1, 11], zeros[1, 4] = 0.0, -0.0
    return dict(q=q, items=items, x=x, mask=mask, vals=vals, zeros=zeros, top2=top2, N=N, D=D)


def _out(vals, k, **kw):
    v, i = SO.exact_topk(vals, k, **kw)
    v, i = v.numpy(), i.numpy()
    return v.astype(np.float32), i, v


def _bounded(w, s, i, d):
    return SO.check_bounded(s, i, d, torch.as_tensor(w["q"]), torch.as_tensor(w["items"]), w["D"], K, w["mask"])


def test_oracle_order_ties_and_signed_zeros(world):
    s, i, d = _out(world["vals"], K)
    assert i[0, 0] < i[0, 1] == world["N"] - 1 and d[0, 0] == d[0, 1]        # tie: lowest id first
    assert world["top2"] not in i[2]
    _, iz, dz = _out(world["zeros"], 3)
    assert iz[1].tolist() == [11, 4, 0] and np.signbit(dz[1, 1]) and not np.signbit(dz[1, 0])  # +0.0, then -0.0
    sv, iv, dv = _out(world["vals"].double(), K)                              # the float64 path agrees
    assert np.array_equal(iv, i) and np.array_equal(dv, d)
    ps, pi, pd = _out(world["vals"][:, :7], K, allow_short=True, id_offset=(1 << 31) + 5)
    assert (pi[:, 7:] == -1).all() and np.isneginf(pd[:, 7:]).all() and (pi[:, :7] >= (1 << 31) + 5).all()


def test_checkers_accept_the_oracle(world):
    s, i, d = _out(world["vals"], K)
    assert SO.check_exact(s, i, d, d, i) == []
    assert _bounded(world, s, i, d) == []


def _mutants(w):
    """(name, s, i, d, flagged by check_bounded too) of wrong outputs."""
    s, i, d = _out(w["vals"], K)
    _, i1, d1 = _out(w["vals"], K + 1)
    out = []

    def mut(name, bounded, f):
        ms, mi, md = s.copy(), i.copy(), d.copy()
        f(ms, mi, md)
        ms = md.astype(np.float32) if name != "float32 score" else ms
        out.append((name, ms, mi, md, bounded))

    r = 3
    assert d[r, K - 1] - d1[r, K] > 1e-2  # far apart: a bound on the summation cannot hide the swap

    def kth(ms, mi, md):
        mi[r, K - 1], md[r, K - 1] = i1[r, K], d1[r, K]

    def tie(ms, mi, md):
        mi[0, [0, 1]] = mi[0, [1, 0]]

    def ulp(ms, mi, md):
        md[1, 4] = np.nextafter(md[1, 4], np.inf)

    def raw(ms, mi, md):  # the masked best item of row 2 back at rank 0 with its raw score
        mi[2, 1:], md[2, 1:] = mi[2, :-1].copy(), md[2, :-1].copy()
        mi[2, 0], md[2, 0] = w["top2"], np.float32(w["x"][2, w["top2"]])

    def order(ms, mi, md):
        mi[3, [2, 3]], md[3, [2, 3]] = mi[3, [3, 2]], md[3, [3, 2]]

    def f32(ms, mi, md):
        ms[1, 0] = np.nextafter(ms[1, 0], np.float32(np.inf))

    mut("k-th replaced by (k+1)-th", True, kth)
    mut("tied ids swapped", True, tie)
    mut("1 ulp", False, ulp)
    mut("masked id with raw score", True, raw)
    mut("out of order", True, order)
    mut("float32 score", True, f32)
    return out


def test_check_exact_flags_every_mutant(world):
    s, i, d = _out(world["vals"], K)
    for name, ms, mi, md, _ in _mutants(world):
        assert SO.check_exact(ms, mi, md, d, i), name
    zs, zi, zd = _out(world["zeros"], K)
    ms, mi, md = zs.copy(), zi.copy(), zd.copy()
    mi[1, [0, 1]], md[1, [0, 1]] = mi[1, [1, 0]], md[1, [1, 0]]
    assert SO.check_exact(ms, mi, md, zd, zi), "+0.0 / -0.0 swapped"
    md2 = zd.copy()
    md2[1, [0, 1]] = md2[1, [1, 0]]  # ids right, signs of the zeros swapped
    assert SO.check_exact(md2.astype(np.float32), zi, md2, zd, zi), "signs of zero swapped"
    ss, si, sd = _out(world["vals"][:, :7], K, allow_short=True)
    mi = si.copy()
    mi[:, -1] = 0
    assert SO.check_exact(ss, mi, sd, sd, si), "padding id missing"
    md = sd.copy()
    md[:, -1] = 0.0
    assert SO.check_exact(md.astype(np.float32), si, md, sd, si), "padding value missing"
    assert SO.check_exact(ss[:, :-1], si[:, :-1], sd[:, :-1], sd, si), "short output"


def test_check_bounded_flags_every_mutant_that_is_not_a_tie(world):
    for name, ms, mi, md, bounded in _mutants(world):
        if bounded:
            assert _bounded(world, ms, mi, md), name


def test_override_emulation_within_gamma_of_float64():
    rs = np.random.RandomState(1)
    for D in (8, 72, 768, 4096):
        for dt in (torch.bfloat16, torch.float16):
            B, N = 6, 50
            q = torch.as_tensor(rs.standard_normal((B, D)).astype(np.float32)).to(dt)
            it = torch.as_tensor(rs.standard_normal((N, D)).astype(np.float32)).to(dt)
            ip = np.array([0, 3, 3, 10, 12, 20, 25])
            cols = np.concatenate([np.sort(rs.choice(N, n, replace=False)) for n in np.diff(ip)]).astype(np.int32)
            vals = rs.standard_normal(25)
            got = SO.override_values(q, it, ip, cols, vals, SO.MASK_ADD, D)
            rows = np.repeat(np.arange(B), np.diff(ip))
            qe, ve = q.double().numpy()[rows], it.double().numpy()[cols]
            exact = (qe * ve).sum(1)
            gamma = D * 2.0 ** -24 / (1 - D * 2.0 ** -24)
            assert (np.abs(got - vals - exact) <= gamma * np.abs(qe * ve).sum(1)).all(), (D, dt)
            assert np.array_equal(SO.override_values(q, it, ip, cols, vals, SO.MASK_SET, D), vals)


def test_override_emulation_follows_the_lane_and_butterfly_order():
    """D = 512: 64 chunks of 8, lane l sums chunks l and l + 32.  Ones in the queries; the item holds 2^24 at
    element 0 (lane 0, chunk 0), 1.0 at element 256 (lane 0, chunk 32) and 1.0 at element 8 l (lane l, chunk
    l) for l = 1..31.  Lane 0: 2^24 + 1 -> 2^24 (ties to even); lanes 1..31: 1.  Butterfly 16: lane 0 2^24 + 1
    -> 2^24, lanes 1..15 2; 8: 2^24 + 2, lanes 1..7 4; 4: 2^24 + 6, 8; 2: 2^24 + 14, 16; 1: 2^24 + 30.  (The
    float64 sum is 2^24 + 32, a sequential fp32 sum 2^24.)"""
    D = 512
    q = np.ones((1, D), dtype=np.float32)
    v = np.zeros((1, D), dtype=np.float32)
    v[0, 0], v[0, 256] = 2.0 ** 24, 1.0
    v[0, 8 * np.arange(1, 32)] = 1.0
    got = SO.override_values(q, v, np.array([0, 1]), np.array([0], np.int32), np.array([0.5]), SO.MASK_ADD, D)
    assert got[0] == 2.0 ** 24 + 30 + 0.5


# ---- the exact plan matrix reaches its branches ----

def _round64(x):
    return (x + 63) // 64 * 64


def _branch_errors(c, plan, want):
    errs = []
    for key in ("algo", "two_cta", "n_q_tiles", "seed_items"):
        if key in want and plan[key] != want[key]:
            errs.append(f"{key} {plan[key]} != {want[key]}")
    if "seeded" in want and (plan["seed_items"] > 0) != want["seeded"]:
        errs.append(f"seeding {plan['seed_items']}")
    if "poller" in want and (plan["algo"] == 2 and plan["n_q_tiles"] >= 32) != want["poller"]:
        errs.append(f"poller: {plan['n_q_tiles']} tiles")
    if "include" in want:
        _, h = mask_args(c, case_mask(c))
        slack = 128 if plan["algo"] == 2 else 32
        cap = _round64(2 * (c["k"] + h) + slack) if want["include"] else _round64(2 * c["k"] + slack)
        if plan["cand_capacity"] != cap:
            errs.append(f"include={want['include']}: capacity {plan['cand_capacity']} != {cap}")
    return errs


@pytest.mark.parametrize("c", CASES, ids=[c["id"] for c in CASES])
def test_plan_matrix_reaches_its_branch(c, lever):
    base = c.get("levers", {})
    if base:
        unset = plan_of(c)
        lever(**base)
        assert plan_of(c) != unset, "the case's levers do not change its plan"
    plan = plan_of(c)
    assert not _branch_errors(c, plan, c["want"]), (plan, _branch_errors(c, plan, c["want"]))
    kept = {key: v for key, v in c["want"].items() if key in ("algo", "seeded", "include")}
    vs = variants(c, plan)
    assert bool(vs) == (plan["algo"] == 2 and (plan["n_q_tiles"] > 1 or plan["seed_items"] > 0 or c["B"] > 128))
    for kv in vs:
        with SO.levers(**kv):
            p2 = plan_of(c)
        assert not _branch_errors(c, p2, kept), (kv, p2)
        if "CCR_LEAD" in kv:
            assert p2["lead_tiles"] == int(kv["CCR_LEAD"]) and p2["two_cta"] == plan["two_cta"]
        if "CCR_2CTA" in kv:
            assert p2["two_cta"] == int(kv["CCR_2CTA"]) != plan["two_cta"]
        if "CCR_NO_HIST" in kv:
            assert p2 == plan  # the histogram switch is not part of plan_info's summary
    assert plan_of(c) == plan


def test_levers_take_effect_and_are_undone(lever):
    from ccr_b200 import _lib

    base = _lib.plan_info(512, 300_000, 64, 10)
    assert base["two_cta"] == 1
    with SO.levers(CCR_2CTA="0", CCR_LEAD="3"):
        p = _lib.plan_info(512, 300_000, 64, 10)
        assert p["two_cta"] == 0 and p["lead_tiles"] == 3
        with SO.levers(CCR_2CTA=None):
            assert _lib.plan_info(512, 300_000, 64, 10)["two_cta"] == 1
        assert _lib.plan_info(512, 300_000, 64, 10)["two_cta"] == 0
    assert _lib.plan_info(512, 300_000, 64, 10) == base and "CCR_2CTA" not in os.environ
    lever(CCR_2CTA="0")
    assert _lib.plan_info(512, 300_000, 64, 10)["two_cta"] == 0


# ---- no test writes a lever behind the library's back ----

# scripts that set levers for a whole run and re-read them themselves
LEVER_SCRIPTS = {"select_oracle.py", "perf_sweep.py", "exact_bench.py", "bm25_bench.py"}


def lever_writes(src, name="<src>"):
    """Environment writes in ``src`` that may set a CCR_* lever: a lever name as the key, or a key that is not
    a literal in a file that names a lever."""
    names_lever = any(lv in src for lv in SO.LEVERS)
    hits = []

    def key(node, line):
        if isinstance(node, ast.Constant) and isinstance(node.value, str):
            if node.value in SO.LEVERS:
                hits.append(f"{name}:{line} {node.value}")
        elif names_lever:
            hits.append(f"{name}:{line} non-literal key")

    def is_environ(n):
        return (isinstance(n, ast.Attribute) and n.attr == "environ") or (isinstance(n, ast.Name) and n.id == "environ")

    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.Call) and isinstance(node.func, ast.Attribute):
            f = node.func
            if f.attr in ("setenv", "delenv", "putenv", "unsetenv") and node.args:
                key(node.args[0], node.lineno)
            elif is_environ(f.value) and f.attr in ("update", "pop", "setdefault", "__setitem__", "__delitem__"):
                for a in node.args:
                    if isinstance(a, ast.Dict):
                        for kn in a.keys:
                            key(kn, node.lineno)
                    elif f.attr == "update" or a is node.args[0]:
                        key(a, node.lineno)
                for kw in node.keywords:
                    key(ast.Constant(kw.arg) if kw.arg else kw.value, node.lineno)
            elif f.attr == "setitem" and node.args and is_environ(node.args[0]) and len(node.args) > 1:
                key(node.args[1], node.lineno)
        targets = node.targets if isinstance(node, (ast.Assign, ast.Delete)) else \
            [node.target] if isinstance(node, ast.AugAssign) else []
        for t in targets:
            if isinstance(t, ast.Subscript) and is_environ(t.value):
                key(t.slice, node.lineno)
    return hits


def test_lever_scan_catches_raw_writes():
    assert lever_writes('monkeypatch.setenv("CCR_2CTA", two)')
    assert lever_writes('os.environ["CCR_LEAD"] = "4"')
    assert lever_writes('env = {"CCR_NO_HIST": "1"}\nos.environ.update(env)')
    assert lever_writes('os.environ.update(CCR_EXACT_FALLBACK="1")')
    assert lever_writes('os.environ.pop("CCR_BM25_BLOCKWIDE", None)')
    assert not lever_writes('monkeypatch.setenv("CCREC_SIM_TYPE", "dot")\nos.environ["CASE_N"] = n')


def test_no_test_sets_a_lever_directly():
    hits = []
    for root, _, files in os.walk(TESTS):
        for fn in files:
            if fn.endswith(".py") and fn not in LEVER_SCRIPTS:
                path = os.path.join(root, fn)
                hits += lever_writes(open(path).read(), os.path.relpath(path, TESTS))
    assert not hits, f"set CCR_* levers through select_oracle.lever / levers (they need a reload): {hits}"
