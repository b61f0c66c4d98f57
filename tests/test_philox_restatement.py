"""The CPU restatement of the device's map generator and random policy (oracle/ngw_oracle.c, last section), checked on
its own: Random123's known answers, the word stream and below(), the reset invariants, and the two rare branches of
the random policy's Lemire draw.  tests/test_gpu_reset_exact.py then compares the GPU with it bit for bit."""
import numpy as np
import pytest

import golden_util
import scenarios
from gym_novel_gridworlds_b200.compiler import compile_chain
from oracle.oracle_lib import OracleBatch, philox4x32_10, philox_below, policy_draw, policy_draws
from test_gpu_reset import _check_base_invariants

C2 = {'env': scenarios.POGO, 'map_size': 10, 'chain': [['limit', scenarios.C2_SET], ['lidar', 8]]}
SEED = 0x5DEECE66D2545F49         # both words non-zero

# Found once with a threaded C search over ngw_oracle.c's ps_block: policy seed SEED, n = 10 actions (C2), gids from
# 0xFFFFF000 upwards, steps 0..15 (2^28 gids x 4 Philox blocks, about 3 s on 8 cores).  The first hits were these two.
LEMIRE_REJECT = (SEED, 0x102255121, 12)      # low half of x * 10 is 2 < (2^32 - 10) mod 10 = 6: continues on 0xFFE
LEMIRE_ACCEPT = (SEED, 0x1004439FF, 7)       # low half 6: enters the test, kept


def _compiled(desc):
    return compile_chain(scenarios.build_chain(scenarios.b200_namespace(), desc))


@pytest.mark.parametrize('ctr,key,want', [
    ([0, 0, 0, 0], [0, 0], [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]),
    ([0xffffffff] * 4, [0xffffffff] * 2, [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]),
    ([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0],
     [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1])])
def test_philox_known_answers(ctr, key, want):
    assert philox4x32_10(ctr, key).tolist() == want


def test_word_stream_is_blocks_in_order():
    """below(0) takes the whole word unmasked: the stream is words 0..3 of block 0, then block 1, ... of counter
    (gid lo, gid hi, episode, stream << 20 | block) under key (seed lo, seed hi).  below(1) consumes nothing."""
    gid, ep, stream = 0x1_2345_6789, 0xFFFFFFFE, 3
    words, used = philox_below(SEED, gid, ep, stream, 0, 12)
    assert used == 12
    blocks = [philox4x32_10([gid & 0xFFFFFFFF, gid >> 32, ep, (stream << 20) | b], [SEED & 0xFFFFFFFF, SEED >> 32])
              for b in range(3)]
    assert words.tolist() == np.concatenate(blocks).tolist()
    assert philox_below(SEED, gid, ep, stream, 1, 50) == (pytest.approx(np.zeros(50)), 0)


@pytest.mark.parametrize('n', [2, 10, 36, 100, 1000, (1 << 20) + 1])
def test_below_is_uniform_and_rejects_at_the_mask_rate(n):
    from scipy.stats import chi2
    count = 200000
    v, used = philox_below(SEED, 77, 5, 1, n, count)
    assert v.max() < n
    mask = (1 << int(n - 1).bit_length()) - 1
    p = n / (mask + 1.0)                                       # acceptance probability of one word
    mean, sd = count / p, np.sqrt(count * (1 - p)) / p          # words used: negative binomial
    assert abs(used - mean) < 6 * sd + 1, (used, mean, sd)
    bins = min(n, 1000)
    hist = np.bincount((v.astype(np.int64) * bins) // n, minlength=bins)
    expect = np.array([((k + 1) * n + bins - 1) // bins - (k * n + bins - 1) // bins for k in range(bins)]) * count / n
    stat = (((hist - expect) ** 2) / expect).sum()
    assert stat < chi2.ppf(1 - 1e-6, bins - 1), stat


def test_restated_resets_keep_the_base_invariants():
    """C2, and AxeHard(iron) whose 11 items crowd the 6x6 interior: envs that reset cleanly have the reference's base
    invariants; on the crowded grid the enumeration fallback runs and some envs flag PLACEMENT."""
    for desc, n in ((C2, 4096), (golden_util.get('pogo_A_axe_hard_iron_inc')['meta'], 8192)):
        cc = _compiled(desc)
        ob = OracleBatch([cc], n)
        flags, obs, ev = ob.reset_philox(SEED, (1 << 32) - n // 2, 0x80000000)
        ok = flags == 0
        _check_base_invariants(cc, ob.map[ok], ob.pose[ok], ob.inv[ok], cc.map_size)
        ob2 = OracleBatch([cc], n)
        ob2.map[:], ob2.pose[:], ob2.inv[:] = ob.map, ob.pose, ob.inv
        assert np.array_equal(ob2.observe(), obs)                       # no ops: the observation is of the final state
        if cc.c.n_place > 2:
            assert ev['place_fail'] > 0 and (~ok).sum() == ev['place_fail'], ev
        else:
            assert ok.all() and ev['fallback'] == 0
        again, _, _ = OracleBatch([cc], n).reset_philox(SEED, (1 << 32) - n // 2, 0x80000000)
        assert np.array_equal(again, flags)


def overfilled(cc):
    """AxeHard(iron) asking for 30 iron: every reset runs out of placeable cells, and on the way down to none, about two
    envs in 10^4 miss the last placeable cell in all 8 side^2 draws and place an item through the enumeration."""
    cc.c.place_qty[list(cc.c.place_item[:cc.c.n_place]).index(cc.item_names.index('iron'))] = 30
    return cc


def test_restated_enumeration_fallback_places_on_placeable_cells():
    cc = overfilled(_compiled(golden_util.get('pogo_A_axe_hard_iron_inc')['meta']))
    n = 100000
    ob = OracleBatch([cc], n)
    flags, _, ev = ob.reset_philox(SEED, 5, 2, want_obs=False)
    assert (flags == 2).all() and ev['place_fail'] == n and ev['fallback'] > 0, ev
    m = ob.map.reshape(n, 10, 10)
    items = (m != 0)
    items[:, [0, -1], :] = False
    items[:, :, [0, -1]] = False
    assert not (items[:, 1:, :] & items[:, :-1, :]).any() and not (items[:, :, 1:] & items[:, :, :-1]).any()
    assert (m[np.arange(n), ob.pose[:, 0], ob.pose[:, 1]] == 0).all()


def test_restated_subset_selection_orders():
    """AddItem on a 40x40 grid (~1000 air candidates, 20-30 %): with the full key the radix-select ends in boundary
    lists or whole bins; with key mask 0 every key ties and the winners are the first `take` candidates in the device's
    arrival order (i >> 7, i & 3, i >> 2) — not in cell order."""
    cc = _compiled(golden_util.get('pogo_ms40_additem_hard')['meta'])
    n = 64
    full = OracleBatch([cc], n)
    _, _, ev = full.reset_philox(SEED, 3, 1)
    assert ev['subset'] == n and ev['list'] > 0 and ev['arrival'] == 0, ev
    tied = OracleBatch([cc], n)
    _, _, ev = tied.reset_philox(SEED, 3, 1, key_mask=0)
    assert ev['arrival'] == n, ev
    spring = cc.c.reset_ops[0].a
    base = OracleBatch([cc], n)
    cfg = base.cfgs[0]
    cfg.n_reset_ops = 0                                          # the same base, without the op
    base.reset_philox(SEED, 3, 1)
    agent = tied.pose[:, 0].astype(int) * 40 + tied.pose[:, 1]
    for e in range(n):
        air = np.nonzero(base.map[e] == 0)[0]
        order = sorted(air, key=lambda i: (i >> 7, i & 3, i >> 2))
        got = set(np.nonzero(tied.map[e] == spring)[0])
        took = len(got) + (1 if agent[e] in order[:len(got) + 1] and agent[e] not in got else 0)
        assert got == set(order[:took]) - {agent[e]}, e
        assert got != set(sorted(air)[:took]) - {agent[e]}, e


def test_random_policy_lemire_branches():
    """The two hard-coded (seed, gid, t) take Lemire's rare branches (probability 6 and 4 in 2^32 per draw for 10
    actions), and the batch draw agrees with the single one there."""
    for case, want in ((LEMIRE_REJECT, 2), (LEMIRE_ACCEPT, 1)):
        seed, gid, t = case
        a, br = policy_draw(seed, gid, t, 10)
        assert br == want and 0 <= a < 10, (case, a, br)
        acts, brs = policy_draws(seed, gid - 5, np.full(9, 10), t + 3)
        assert acts[t, 5] == a and brs[t, 5] == want
        assert (brs[:, [0, 1, 2, 3, 4, 6, 7, 8]] == 0).all() and (brs[:t, 5] == 0).all() and (brs[t + 1:, 5] == 0).all()
    acts, brs = policy_draws(SEED, (1 << 32) - 100, np.arange(200) % 16 + 1, 40)
    assert (acts >= 0).all() and (acts < (np.arange(200) % 16 + 1)[None, :]).all()
    one = np.array([[policy_draw(SEED, (1 << 32) - 100 + e, t, e % 16 + 1)[0] for e in range(200)] for t in range(40)])
    assert np.array_equal(one, acts)
