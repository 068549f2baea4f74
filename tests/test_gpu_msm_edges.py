"""GPU: the MSM at every window width, on the signed recoding's edge scalars, and on inputs that drive the group law's
exceptional branches (P + P, P + (-P), infinity operands) through every stage of the pipeline — k_accumulate, the three
merge kernels, the three reduction-tree kernels and the host's Horner pass over the window sums — in G1 and G2, with
and without a window table, and in batched-affine mode.

Every expected value is a closed form: the bases are k_i * G with known k_i (made on the GPU by the fixed-base kernel,
k_i = 0 giving infinity and r - k giving the negation), so sum s_i P_i = (sum k_i s_i mod r) * G, computed by
oracle/bn254.py.  Outputs are compared limb for limb.  Which branch a construction reaches is shown with the CPU models
of tests/test_msm_digits_cpu.py (recoding, task split, reduction tree) before it runs.
"""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import bn254 as bn
from oracle.bn254 import R
from tests.test_msm_digits_cpu import (boundary_scalars, k_digits, merge_class, msm_num_windows, pick_seg,
                                       reduce_tree, tail_l0)

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SWEEP_N = 256
FORCED = 12        # the forced width of the constructions: levels 2 and 3 of the tree run in k_reduce_level


@pytest.fixture(scope="module")
def ectx():
    """A context of this module's own: its workspaces grow to ~20 GB at c = 22 and are released with it."""
    from gnark_whir_b200 import lib
    c = lib.Context(0)
    yield c
    c.close()


def _gen(group):
    return bn.g1_to_array([bn.G1_GEN])[0] if group == 1 else bn.g2_to_array([bn.G2_GEN])[0]


def _closed(group, ks, ss):
    dot = sum(k * s for k, s in zip(ks, ss)) % R
    return bn.g1_to_array([bn.g1_mul(bn.G1_GEN, dot)])[0] if group == 1 else bn.g2_to_array([bn.g2_mul(bn.G2_GEN, dot)])[0]


def _bases(ctx, group, ks):
    return ctx.fixed_base_mul(_gen(group), bn.fr_to_mont_array([k % R for k in ks]), group=group, resident=True)


def _check(ctx, group, ks, ss, c=0, table=None, offset=0, n=None):
    """MSM over k_i G with scalars s_i, plain at width c (0 = automatic) or through a window table of width `table`
    (0 = automatic), over points [offset, offset + n); compared with the closed form.  Returns the width used."""
    n = len(ks) - offset if n is None else n
    bases = _bases(ctx, group, ks)
    try:
        if table is not None:
            used = bases.precompute(table)
            assert used == table or table == 0
        ctx.set_msm_window(c)
        cu, W = ctx.msm_plan(bases, n)
        out = ctx.msm(bases, bn.fr_to_mont_array(ss[offset:offset + n]), offset=offset)
    finally:
        ctx.set_msm_window(0)
        bases.free()
    exp = _closed(group, ks[offset:offset + n], ss[offset:offset + n])
    assert np.array_equal(out, exp), (group, c, table, cu)
    assert W == msm_num_windows(cu)
    return cu


def _width(ctx, group, n, c, table):
    """The window width an n-point MSM in this mode runs at."""
    bases = _bases(ctx, group, [1] * n)
    try:
        if table is not None:
            return bases.precompute(table)
        ctx.set_msm_window(c)
        return ctx.msm_plan(bases, n)[0]
    finally:
        ctx.set_msm_window(0)
        bases.free()


def _sweep_inputs(rng, c, n=SWEEP_N):
    ss = [s for _, s in boundary_scalars(c, msm_num_windows(c))]
    ss += [rng.randrange(R) for _ in range(n - len(ss))]
    ks = [rng.randrange(1, R) for _ in range(n)]
    return ks, ss


# ---- 1. plain window widths: every c the API accepts for G1 up to 22, G2 up to 20.  G2 above c = 20 would need
# about 145 GB of workspace (256-byte buckets in three rotating sets) and is not run.
@pytest.mark.parametrize("group,c", [(1, c) for c in range(2, 23)] + [(2, c) for c in range(2, 21)])
def test_msm_plain_every_width(ectx, group, c):
    rng = random.Random(1000 * group + c)
    ks, ss = _sweep_inputs(rng, c)
    assert _check(ectx, group, ks, ss, c=c) == c


# ---- 2. G1 at c = 23 and 24 (nb = 11 * 2^23 buckets: ~75 GB of workspace) in a context of its own
@pytest.mark.parametrize("c", [23, 24])
def test_msm_g1_widest_windows(c):
    import torch
    from gnark_whir_b200 import lib
    free, _ = torch.cuda.mem_get_info()
    if free < 90e9:
        pytest.skip(f"c = {c} needs ~75 GB of workspace; {free / 1e9:.1f} GB free")
    rng = random.Random(c)
    ks, ss = _sweep_inputs(rng, c)
    big = lib.Context(0)
    try:
        assert _check(big, 1, ks, ss, c=c) == c
    finally:
        big.close()


# ---- 3. window tables: every width for G1, four for G2; whole vector and a sub-range
@pytest.mark.parametrize("group,c", [(1, c) for c in range(8, 23)] + [(2, c) for c in (8, 12, 16, 20)])
def test_msm_table_every_width(ectx, group, c):
    rng = random.Random(5000 + 1000 * group + c)
    ks, ss = _sweep_inputs(rng, c)
    assert _check(ectx, group, ks, ss, table=c) == c
    assert _check(ectx, group, ks, ss, table=c, offset=37, n=150) == c


# ---- 5. exceptional branches.  Modes: automatic / forced plain width, automatic / forced table width.
MODES = {"auto": (0, None), "c12": (FORCED, None), "table-auto": (0, 0), "table12": (0, FORCED)}
TARGET_PER_SM = 2048          # msm_enqueue: target_tasks = SMs * 2048


def _sm_target():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * TARGET_PER_SM


def _buckets(ks, ss, c, table):
    """Bucket values as discrete logs (0 = infinity): one list per window, or the one shared set of a table."""
    W = msm_num_windows(c)
    nbw = 1 << (c - 1)
    sets = [[0] * nbw for _ in range(1 if table else W)]
    for k, s in zip(ks, ss):
        d, _ = k_digits(s % R, c, W)
        for w, x in enumerate(d):
            if x:
                row = (k << (c * w)) if table else k      # a table's row w holds 2^(cw) P
                b = sets[0 if table else w]
                b[abs(x) - 1] = (b[abs(x) - 1] + (row if x > 0 else -row)) % R
    return sets


def _tree_kinds(ks, ss, c, table):
    """Addition kinds each reduction kernel meets, over all windows (CPU replay of the tree)."""
    seen = {}
    for B in _buckets(ks, ss, c, table):
        _, s = reduce_tree(B, c, tail_l0(c))
        for kern, kinds in s.items():
            seen.setdefault(kern, set()).update(kinds)
    return seen


def _same_point(n, rng):
    k = rng.randrange(1, R)
    return [k] * n, [1] * n


def _one_per_bucket(c, n, rng, table=False):
    """n >= 2^(c-1) copies of P; s_i = i + 1 puts one P in each of window 0's buckets 0 .. nbw - 2.  Bucket nbw - 1
    is digit -nbw: base -P with scalar nbw puts -(-P) = P there too (and -P into bucket 0 of window 1).  Through a
    table that window-1 entry is -2^c P in the one shared bucket 0; a base 2^c P with scalar 1 cancels it there."""
    nbw = 1 << (c - 1)
    k = rng.randrange(1, R)
    ks = [k] * (nbw - 1) + [R - k] + [k] * (n - nbw)
    ss = list(range(1, nbw)) + [nbw] + [0] * (n - nbw)
    if table:
        ks[-1], ss[-1] = (k << c) % R, 1
    return ks, ss


def _alternating(n, rng):
    k, s = rng.randrange(1, R), rng.randrange(1, R)
    return [k, R - k] * (n // 2), [s] * n


def _tree_cancel(c, rng):
    """Window-0 buckets b and b + 2^(n - m) (n = c - 1) meet first at level m of the tree; holding P_m and -P_m they
    cancel there, and the infinity they leave is an operand at every later level and in the tail's final sum.  One
    such pair per level m = 1 .. n where a free pair of buckets is left (all levels from c = 5 up)."""
    nbw = 1 << (c - 1)
    used = set()
    ks, ss = [], []
    for m in range(1, c):
        step = nbw >> m
        # b and b + step meet at level m when b mod 2 step < step; bucket nbw - 1 (digit -nbw) is left out
        x = next((b for b in range(nbw - 1 - step) if b % (2 * step) < step and not {b, b + step} & used), None)
        if x is None:          # narrow widths: no free pair for this level
            continue
        used |= {x, x + step}
        k = rng.randrange(1, R)
        ks += [k, R - k]
        ss += [x + 1, x + step + 1]            # digit b + 1 addresses bucket b
    return ks, ss


def _horner_cancel(c, rng):
    """Window sums that cancel in the host's Horner pass: G at window j + 1 and -(2^c) G at window j, then a third
    point in window 0 after the infinity.  (Through a table both land in one bucket and cancel in k_accumulate.)"""
    W = msm_num_windows(c)
    j = W // 2
    q = rng.randrange(1, R)
    return [1, R - (1 << c), q, 1, R - (1 << c)], [1 << (c * (j + 1)), 1 << (c * j), 3, 1 << c, 1]


def _infinity_heavy(n, rng):
    """Every third base is infinity, all scalars 1: infinity entries all through one heavy bucket."""
    ks = [0 if i % 3 == 1 else rng.randrange(1, R) for i in range(n)]
    return ks, [1] * n


def _table_rows(c, rng):
    """Bases P and 2^c P with scalars d 2^c and d: through a width-c table P's row 1 and 2^c P's row 0 put the same
    point into bucket d - 1 (a doubling in k_accumulate); with -2^c P they cancel.  Without a table the two land in
    windows 1 and 0, and the Horner pass adds equal (and opposite) window sums."""
    ks, ss = [], []
    for _ in range(8):
        k, d = rng.randrange(1, R), rng.randrange(1, 1 << (c - 1))
        ks += [k, (k << c) % R, k, R - ((k << c) % R)]
        ss += [d << c, d, d << c, d]
    return ks, ss


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("n,cls", [(96, "k_merge_pass"), (320, "k_merge_mid"), (2048, "k_merge_heavy")])
def test_same_point_all_ones(ectx, group, mode, n, cls):
    """One point, n copies, scalar 1: every task's second entry takes madd's doubling branch, and its equal task
    partials meet in the merge class named by `cls` (seg = 32: 3, 10 and 64 tasks)."""
    c, table = MODES[mode]
    cu = _width(ectx, group, n, c, table)
    nb = (1 << (cu - 1)) * (1 if table is not None else msm_num_windows(cu))
    seg = pick_seg(n, nb, _sm_target())
    assert merge_class(-(-n // seg)) == cls
    ks, ss = _same_point(n, random.Random(n + group))
    _check(ectx, group, ks, ss, c=c, table=table)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_one_point_per_bucket(ectx, group, mode):
    """Every bucket of window 0 holds the same P: every level of k_reduce_first / _level / _tail adds equal values."""
    c, table = MODES[mode]
    n = 2048
    cu = _width(ectx, group, n, c, table)
    ks, ss = _one_per_bucket(cu, n, random.Random(group), table is not None)
    kinds = _tree_kinds(ks, ss, cu, table is not None)
    assert "dbl" in kinds["k_reduce_first"] and "dbl" in kinds["k_reduce_tail"]
    if tail_l0(cu) > 2:
        assert "dbl" in kinds["k_reduce_level"]
    _check(ectx, group, ks, ss, c=c, table=table)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_alternating_p_minus_p(ectx, group, mode):
    """P, -P, P, -P, ... with one scalar: each bucket's accumulation cancels to infinity in madd and restarts from it;
    the result is infinity (64 tasks per bucket: the heavy merge adds infinities)."""
    c, table = MODES[mode]
    ks, ss = _alternating(2048, random.Random(group))
    _check(ectx, group, ks, ss, c=c, table=table)
    assert _closed(group, ks, ss).sum() == 0


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_tree_cancellation(ectx, group, mode):
    """Buckets P_m and -P_m that meet at level m of the tree, for every level: cancellations in k_reduce_first,
    k_reduce_level (forced width) and k_reduce_tail, and infinity operands after them."""
    c, table = MODES[mode]
    cu = _width(ectx, group, 2 * (FORCED - 1), c, table)
    ks, ss = _tree_cancel(cu, random.Random(group))
    kinds = _tree_kinds(ks, ss, cu, table is not None)
    assert "cancel" in kinds["k_reduce_first"] and "cancel" in kinds["k_reduce_tail"]
    assert kinds["k_reduce_tail"] & {"q_inf", "self_inf"}
    if tail_l0(cu) > 2:
        assert "cancel" in kinds["k_reduce_level"] and kinds["k_reduce_level"] & {"q_inf", "self_inf"}
    assert _check(ectx, group, ks, ss, c=c, table=table) == cu


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_horner_window_sums_cancel(ectx, group, mode):
    c, table = MODES[mode]
    cu = _width(ectx, group, 5, c, table)
    ks, ss = _horner_cancel(cu, random.Random(group))
    _check(ectx, group, ks[3:], ss[3:], c=c, table=table)            # G, -(2^c) G with 2^c, 1: infinity
    assert _closed(group, ks[3:], ss[3:]).sum() == 0
    _check(ectx, group, ks, ss, c=c, table=table)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_infinity_bases(ectx, group, mode):
    c, table = MODES[mode]
    rng = random.Random(group)
    ks, ss = _infinity_heavy(2048, rng)
    _check(ectx, group, ks, ss, c=c, table=table)
    _check(ectx, group, [0] * 300, [rng.randrange(R) for _ in range(300)], c=c, table=table)   # all infinity


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("group", [1, 2])
def test_table_rows_coincide(ectx, group, mode):
    c, table = MODES[mode]
    cu = _width(ectx, group, 32, c, table)
    ks, ss = _table_rows(cu, random.Random(group))
    _check(ectx, group, ks, ss, c=c, table=table)


# ---- 6. batched-affine accumulation on the heaviest constructions
@pytest.fixture
def affine_ectx(ectx):
    from gnark_whir_b200 import lib
    ectx.set_msm_batch_affine(2, 4, 1)
    try:
        yield ectx
    finally:
        ectx.set_msm_batch_affine(*lib.MSM_BATCH_AFFINE_DEFAULT)


@pytest.mark.parametrize("mode", ["auto", "table12"])
@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("build", [_same_point, _alternating, _infinity_heavy])
def test_batch_affine_constructions(affine_ectx, group, mode, build):
    c, table = MODES[mode]
    ks, ss = build(2048, random.Random(group))
    _check(affine_ectx, group, ks, ss, c=c, table=table)


# ---- 7. the other two reduction variants (B200G16_REDUCE_INLINE is read once per process: a child process each)
REDUCE_SUBSET_WIDTHS = (2, 3, 4, 9, 16, 20)


def _reduce_variant_main():
    """G1 width subset, one point per bucket and tree cancellation, against the closed forms; raises on a mismatch."""
    from gnark_whir_b200 import lib
    ctx = lib.Context(0)
    try:
        for c in REDUCE_SUBSET_WIDTHS:
            ks, ss = _sweep_inputs(random.Random(c), c)
            assert _check(ctx, 1, ks, ss, c=c) == c
        ks, ss = _one_per_bucket(FORCED, 2048, random.Random(3))
        _check(ctx, 1, ks, ss, c=FORCED)
        ks, ss = _tree_cancel(FORCED, random.Random(4))
        _check(ctx, 1, ks, ss, c=FORCED)
    finally:
        ctx.close()
    print("reduce variant ok")


@pytest.mark.parametrize("variant", ["0", "1"])
def test_reduce_inline_variants(variant):
    env = dict(os.environ, B200G16_REDUCE_INLINE=variant)
    code = "import tests.test_gpu_msm_edges as t; t._reduce_variant_main()"
    out = subprocess.run([sys.executable, "-c", code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "reduce variant ok" in out.stdout, (out.stdout + out.stderr)[-3000:]
