"""Position-specific template profiles (aadp_set_profile_scoring), CPU side: the oracle construction the GPU tests of
tests/test_gpu_profile.py rely on, and the Python packing of the profiles.

A profile scores sim(i, j) = prof[t][j-1, q_i].  The GPU results are compared with the oracle's table-driven fill
(fill_tab) over the dense similarity matrix of the profile and the uniform affine gap tables of the align type.  That
construction is checked here first: with the identity profile prof[t][j-1, a] = sub[a, t_j] it must reproduce the
substitution fill Oracle.fill exactly, in all five modes and both directions."""
import numpy as np
import pytest

from util import po, MODES, MODE_NAMES, assert_matrix_equal
from test_scoring_space import asym_matrix, dyadic_matrix, seq

MODE_IDS = [MODE_NAMES[m] for m in MODES]


# ---- helpers shared with tests/test_gpu_profile.py ----

def identity_profile(sub, t):
    """prof[j-1, a] = sub[a, t_j]: the profile that scores exactly like the substitution matrix."""
    return np.ascontiguousarray(np.asarray(sub, np.float32)[:, np.asarray(t, np.int64)].T)


def profile_sim(prof, q):
    """(Lq+2, Lt+2) SimilarityMatrix of a profile: interior sim[i, j] = prof[j-1, q_i], borders 0."""
    q = np.asarray(q, np.int64)
    prof = np.asarray(prof, np.float32)
    s = np.zeros((len(q) + 2, prof.shape[0] + 2), np.float32)
    if len(q) and prof.shape[0]:
        s[1:-1, 1:-1] = prof[:, q].T
    return s


def affine_tables(Lq, Lt, gi, ge, at):
    """del_tab / ins_tab of include/aadp.h (aadp_fill_pair_tabulated) for gap(len) = gi + ge*(len-1) in fp32 with the
    free end gaps of align type `at` (aasubalib.h:27-77)."""
    f32 = np.float32
    sz1, sz2 = Lq + 2, Lt + 2
    del_free = at in (po.LOCAL, po.SEMI_LOCAL, po.LOCAL_GLOBAL)
    ins_free = at in (po.LOCAL, po.SEMI_LOCAL, po.GLOBAL_LOCAL)

    def pen(n):
        return (f32(gi) + (f32(ge) * (np.asarray(n) - 1).astype(f32)).astype(f32)).astype(f32)

    t1, t2 = np.meshgrid(np.arange(sz2), np.arange(sz2), indexing="ij")
    dt = np.where(t2 >= t1 + 2, pen(t2 - t1 - 1), f32(0)).astype(f32)
    if del_free:
        dt[(t1 == 0) | (t2 == sz2 - 1)] = 0
    ln, c2 = np.meshgrid(np.arange(sz1 - 1), np.arange(sz2), indexing="ij")
    it = np.where((ln >= 1) & (c2 >= 1), pen(np.maximum(ln, 1)), f32(0)).astype(f32)
    if ins_free:
        it[(c2 == 1) | (c2 == sz2 - 1)] = 0
    return dt, it


def profile_fill(prof, q, gi, ge, at, direction):
    """The oracle's fill of one pair under a profile: (score, prev_q, prev_t, sim)."""
    sim = profile_sim(prof, q)
    dt, it = affine_tables(len(q), prof.shape[0], gi, ge, at)
    s, pq, pt = po.Oracle.fill_tab(sim, dt, it, at == po.LOCAL, direction, True)
    return s, pq, pt, sim


def random_profile(rng, L, A, kind):
    """Seeded position-specific profiles: 'int127' integers up to +/-127 (both ends present), 'grid3' multiples of
    2^-3, 'ties' +/-1."""
    if kind == "int127":
        p = rng.integers(-127, 128, (L, A)).astype(np.float32)
        if L:
            p[0, 0], p[-1, A - 1] = 127, -127
    elif kind == "grid3":
        p = (rng.integers(-80, 81, (L, A)) / 8.0).astype(np.float32)
    else:
        p = rng.choice([-1.0, 1.0], (L, A)).astype(np.float32)
    return p


# ---- the oracle construction ----

@pytest.mark.parametrize("at", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("A,gi,ge", [(1, 3.0, 1.0), (20, 7.0, 2.0), (33, 4.0, 0.0), (64, 0.0, 0.0), (20, 3.0 + 1 / 256.0, 0.5)])
def test_identity_profile_tables_reproduce_the_substitution_fill(A, gi, ge, at):
    sub = dyadic_matrix(A, 300 + A) if gi != int(gi) else asym_matrix(A, 300 + A)
    O = po.Oracle(sub, gi, ge, at)
    rng = np.random.default_rng(17 * A + at)
    for Lq, Lt in [(0, 0), (0, 5), (4, 0), (1, 1), (1, 9), (9, 1), (13, 17), (31, 24)]:
        q, t = seq(rng, Lq, A), seq(rng, Lt, A)
        for d in (po.FWD, po.REV):
            want = O.fill(q, t, d, True)
            got = profile_fill(identity_profile(sub, t), q, gi, ge, at, d)
            for name, g, w in zip(("score", "prevq", "prevt"), got[:3], want):
                assert_matrix_equal("A%d at%d %dx%d d%d %s" % (A, at, Lq, Lt, d, name), g, w)
            assert_matrix_equal("sim", got[3], O.sim(q, t))


def test_profile_tables_see_the_template_position():
    # a profile that differs from the identity at one template position changes the oracle's optimum: the construction
    # really is position specific
    A, at = 4, po.GLOBAL
    sub = asym_matrix(A, 5)
    rng = np.random.default_rng(3)
    q, t = seq(rng, 12, A), seq(rng, 12, A)
    p = identity_profile(sub, t)
    s0 = profile_fill(p, q, 4.0, 1.0, at, po.FWD)[0][-1, -1]
    p[5, :] += 50
    s1 = profile_fill(p, q, 4.0, 1.0, at, po.FWD)[0][-1, -1]
    assert s1 > s0


# ---- packing of Context.set_profile_scoring ----

def test_pack_profiles_offsets_and_empty_profiles():
    from alignment_algos_b200.api import Context
    a = np.arange(6, dtype=np.float32).reshape(3, 2)
    b = np.full((1, 2), -1.5, np.float32)
    prof, off, A = Context.pack_profiles([None, a, np.zeros((0, 2)), b, None])
    assert A == 2
    assert off.dtype == np.int64 and list(off) == [0, 0, 6, 6, 8, 8]
    assert prof.dtype == np.float32 and prof.flags["C_CONTIGUOUS"]
    assert list(prof) == [0, 1, 2, 3, 4, 5, -1.5, -1.5]
    # profile s is prof[off[s]:off[s+1]], row-major (L, A)
    assert np.array_equal(prof[off[1]:off[2]].reshape(-1, A), a)


def test_pack_profiles_refuses_mixed_or_missing_alphabets():
    from alignment_algos_b200.api import Context
    with pytest.raises(ValueError):
        Context.pack_profiles([np.zeros((2, 3)), np.zeros((2, 4))])
    with pytest.raises(ValueError):
        Context.pack_profiles([None, None])
    with pytest.raises(ValueError):
        Context.pack_profiles([np.zeros(5)])
