"""CPU model of the MSM's scalar recoding (csrc/msm_common.cu) and bucket-reduction schedule (csrc/msm_impl.cuh).

`msm_num_windows` and `k_digits` are restated line for line, with the kernel's names, and checked against what a
signed-digit recoding has to do for every window width the API accepts (c = 2..24): the digits sum back to the
scalar, each digit is in [-2^(c-1), 2^(c-1) - 1], no carry leaves the top window, and W is the fewest windows that
allows that.  `boundary_scalars` builds, per (c, W), the scalars that sit on the recoding's edges; the GPU tests in
test_gpu_msm_edges.py feed them to the kernels.  `reduce_tree` replays k_reduce_first / _level / _tail on discrete
logarithms, so the GPU tests' constructions can be shown here, without a GPU, to reach the group law's doubling and
cancelling branches at the levels they claim.
"""
import random

import pytest

from oracle.bn254 import R

MASK64 = (1 << 64) - 1
RM1 = R - 1
WIDTHS = range(2, 25)


# ---- msm_common.cu, restated
def shr256(v, s):  # low 64 bits of v >> s
    if s >= 256:
        return 0
    return (v >> s) & MASK64


def msm_num_windows(c):
    W = (254 + c - 1) // c
    # the top window must absorb the carry of the signed recoding without overflowing
    top = shr256(RM1, (W - 1) * c) + 1
    if top >= (1 << (c - 1)):
        W += 1
    return W


def k_digits(s, c, W):
    """Signed digits of canonical s exactly as k_digits produces them, and the carry left after window W - 1."""
    limbs = [(s >> (32 * k)) & 0xFFFFFFFF for k in range(8)] + [0]
    mask = (1 << c) - 1
    half = 1 << (c - 1)
    carry = 0
    digits = []
    for w in range(W):
        bit = w * c
        q, r = bit >> 5, bit & 31
        raw = 0
        if q < 8:
            two = limbs[q] | (limbs[q + 1] << 32)
            raw = (two >> r) & mask
        raw += carry
        if raw >= half:
            d, carry = raw - (1 << c), 1
        else:
            d, carry = raw, 0
        digits.append(d)
    return digits, carry


def raw_windows(s, c, W):
    """(raw window field, carry into the window) per window: the `raw` and `carry` k_digits adds."""
    out, carry = [], 0
    for w in range(W):
        raw = (s >> (w * c)) & ((1 << c) - 1)
        out.append((raw, carry))
        carry = 1 if raw + carry >= 1 << (c - 1) else 0
    return out


def top_reach(c, W):
    """Largest raw + carry any s < r puts into window W - 1.  The carry out of the windows below is monotone in the
    scalar's low bits, so it is r - 1's (for the largest top field) or T - 1 plus a carry = T below that."""
    k = (W - 1) * c
    T = RM1 >> k
    raw, carry = raw_windows(RM1, c, W)[W - 1]
    return max(raw + carry, T)


# ---- boundary scalars per (c, W): every one below r, each asserted to hit its edge
def boundary_scalars(c, W):
    half = 1 << (c - 1)
    out = [("zero", 0), ("one", 1), ("two", 2), ("r-1", R - 1), ("r-2", R - 2),
           ("half-1", half - 1), ("half", half), ("half+1", half + 1), ("2^c-1", (1 << c) - 1), ("2^c", 1 << c)]
    # window 0 at the edges of the digit range: half - 1 stays positive, half flips to -half with a carry
    assert k_digits(half - 1, c, W)[0][0] == half - 1
    assert k_digits(half, c, W)[0][:2] == [-half, 1]
    assert k_digits((1 << c) - 1, c, W)[0][:2] == [-1, 1]

    # every window's raw field exactly half: window 0 gives -half, every later one half + 1 (carry in) -> -(half - 1)
    K = W
    while True:
        s = sum(half << (c * w) for w in range(K))
        if s < R:
            break
        K -= 1
    d, _ = k_digits(s, c, W)
    assert d[0] == -half and all(x == -(half - 1) for x in d[1:K]) and K >= W - 2
    out.append(("raw-half-every-window", s))

    # every digit exactly -half: raw + carry = half in every window, a carry through every window
    K = W
    while True:
        s = (1 << (c * K)) - half * sum(1 << (c * w) for w in range(K))
        if s < R:
            break
        K -= 1
    d, _ = k_digits(s, c, W)
    assert all(x == -half for x in d[:K]) and d[K] == 1 and K >= W - 2
    out.append(("digit-minus-half-every-window", s))

    # every window all ones: window 0 -> -1, then raw + carry = 2^c -> digit 0 and a carry out, up to the top
    K = 253 // c
    s = (1 << (c * K)) - 1
    d, _ = k_digits(s, c, W)
    assert s < R and d[0] == -1 and all(x == 0 for x in d[1:K]) and d[K] == 1 and K >= W - 2
    out.append(("all-ones-every-window", s))

    # a carry into the top scalar window (the last one 254 bits need) with that window as large as it gets
    Wt = (254 + c - 1) // c - 1
    k = Wt * c
    T = RM1 >> k
    cand = RM1 if raw_windows(RM1, c, W)[Wt][1] else (T << k) - 1
    raw, carry = raw_windows(cand, c, W)[Wt]
    assert carry == 1 and raw + carry >= T
    out.append(("carry-into-top", cand))

    if W > Wt + 1 and top_reach(c, Wt + 1) >= half:
        # W was bumped and a scalar below r reaches the extra window: r - 1 does (see test_num_windows_minimal)
        d, _ = k_digits(RM1, c, W)
        assert d[W - 1] == 1
        out.append(("reaches-extra-window", RM1))
    assert all(0 <= s < R for _, s in out)
    return out


# ---- k_pick_seg and k_tasks' merge classes
def pick_seg(total, nb, target):
    a, b = 2 * (total // nb) + 2, total // target + 1
    seg = a if (nb >= target // 2 and a > b) else b
    return max(seg, 32)


def merge_class(ntasks):
    """Which kernel finishes a bucket split into ntasks tasks (k_tasks)."""
    if ntasks <= 1:
        return "none"
    if ntasks <= 4:
        return "k_merge_pass"
    return "k_merge_mid" if ntasks <= 16 else "k_merge_heavy"


# ---- the reduction tree of one window, on discrete logs (0 = infinity)
def _kind(a, b):
    if b == 0:
        return "q_inf"
    if a == 0:
        return "self_inf"
    if a == b:
        return "dbl"
    if (a + b) % R == 0:
        return "cancel"
    return "add"


def reduce_tree(B, c, l0):
    """Replay k_reduce_first, k_reduce_level (levels < l0) and k_reduce_tail over bucket values B (len 2^(c-1)).
    Returns (sum_b (b + 1) B_b mod r, {kernel: set of addition kinds})."""
    nbw, n = len(B), c - 1
    assert nbw == 1 << n
    seen = {"k_reduce_first": set(), "k_reduce_level": set(), "k_reduce_tail": set()}
    A = list(B)
    half = nbw >> 1
    for i in range(half):
        seen["k_reduce_first"].add(_kind(B[i], B[i + half]))
        A[i] = (B[i] + B[i + half]) % R
    for l in range(2, n + 1):
        s = nbw >> l
        where = "k_reduce_level" if l < l0 else "k_reduce_tail"
        for j in range(l):
            for i in range(s):
                p = (nbw >> j if j else 0) + i
                seen[where].add(_kind(A[p], A[p + s]))
                A[p] = (A[p] + A[p + s]) % R
    for t in range(1, n):
        A[1 << t] = (A[1 << t] << t) % R
    slot = lambda idx: 0 if idx == 0 else 1 << (idx - 1)
    length = n + 1
    while length > 1:
        h = (length + 1) >> 1
        for t in range(length - h):
            seen["k_reduce_tail"].add(_kind(A[slot(t)], A[slot(t + h)]))
            A[slot(t)] = (A[slot(t)] + A[slot(t + h)]) % R
        length = h
    return A[0], seen


def tail_l0(c):
    """First level the one-CTA tail kernel takes (msm_enqueue)."""
    nlev, nbw, l0 = c - 1, 1 << (c - 1), 1
    while l0 <= nlev and l0 * (nbw >> l0) > 512:
        l0 += 1
    return max(l0, 2)


# ---------------------------------------------------------------------------------------------------- tests
def _scalars(c, W, rng):
    return [s for _, s in boundary_scalars(c, W)] + [rng.randrange(R) for _ in range(64)]


@pytest.mark.parametrize("c", WIDTHS)
def test_digits_recompose_in_range_no_carry_out(c):
    rng = random.Random(c)
    W = msm_num_windows(c)
    half = 1 << (c - 1)
    for s in _scalars(c, W, rng):
        d, carry = k_digits(s, c, W)
        assert carry == 0, (c, s)
        assert all(-half <= x <= half - 1 for x in d), (c, s)
        assert sum(x << (c * w) for w, x in enumerate(d)) == s, (c, s)


@pytest.mark.parametrize("c", WIDTHS)
def test_num_windows_covers_every_scalar(c):
    """No s < r carries out of window W - 1: the largest raw + carry the top window can see stays below 2^(c-1)."""
    W = msm_num_windows(c)
    assert top_reach(c, W) < 1 << (c - 1)
    assert W * c >= 254


@pytest.mark.parametrize("c", WIDTHS)
def test_num_windows_minimal(c):
    """W - 1 windows lose r - 1: its recoding no longer sums back.  c = 3 is the one width where the rule is one
    window generous: its bound ((r - 1) >> 252) + 1 = 4 = 2^(c-1) assumes a carry into window 84 on top of the
    field's largest value 3, but every s < r with that field has zeros in window 83 (r - 1 has bits 251..248 clear),
    so no carry reaches it and window 85 is always empty.  Harmless (86 windows of which one holds no entries)."""
    W = msm_num_windows(c)
    d, carry = k_digits(RM1, c, W - 1)
    lost = carry != 0 or sum(x << (c * w) for w, x in enumerate(d)) != RM1
    if c == 3:
        assert not lost and top_reach(c, W - 1) < 1 << (c - 1)
    else:
        assert lost


def test_num_windows_bumped_widths():
    """Only c = 2 and c = 3 take the extra window; at c = 2, W = 128 sits at the library's 128-window limit."""
    bumped = {c: msm_num_windows(c) for c in WIDTHS if msm_num_windows(c) != (254 + c - 1) // c}
    assert bumped == {2: 128, 3: 86}
    d, _ = k_digits(RM1, 2, 128)
    assert d[127] == 1          # r - 1 needs it at c = 2


@pytest.mark.parametrize("c", WIDTHS)
def test_boundary_scalars_build(c):
    names = [n for n, _ in boundary_scalars(c, msm_num_windows(c))]
    assert ("reaches-extra-window" in names) == (c == 2)


@pytest.mark.parametrize("c", [2, 3, 4, 7, 12])
def test_reduce_tree_model_matches_weighted_sum(c):
    rng = random.Random(c)
    nbw = 1 << (c - 1)
    B = [0 if rng.random() < 0.3 else rng.randrange(1, R) for _ in range(nbw)]
    got, _ = reduce_tree(B, c, tail_l0(c))
    assert got == sum((b + 1) * x for b, x in enumerate(B)) % R


def test_pick_seg_classes():
    target = 148 * 2048
    assert pick_seg(96, 64 * 8, target) == 32 and merge_class(3) == "k_merge_pass"
    assert [merge_class(n) for n in (1, 2, 4, 5, 16, 17)] == ["none", "k_merge_pass", "k_merge_pass", "k_merge_mid",
                                                              "k_merge_mid", "k_merge_heavy"]
