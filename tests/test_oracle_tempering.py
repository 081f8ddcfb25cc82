"""The C oracle's temperature ladders (oracle/me_oracle_ladder.c, meo_run_ladder): the replica-exchange uniform against an
independent Philox4x32-7, the equilibrium each rung samples, and the deterministic even/odd count of swap attempts that
``MetropolisEngine.swap_acceptance_rate`` divides by."""
import numpy as np
import pytest


def philox4x32_7(c, k):
    M = 0xFFFFFFFF
    c, k = list(c), list(k)
    for _ in range(7):
        p0, p1 = 0xD2511F53 * c[0], 0xCD9E8D57 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k[0]) & M, p1 & M, ((p0 >> 32) ^ c[3] ^ k[1]) & M, p0 & M]
        k = [(k[0] + 0x9E3779B9) & M, (k[1] + 0xBB67AE85) & M]
    return c


@pytest.mark.parametrize("seed,chain,n", [(0, 0, 1), (5, 17, 2), (2 ** 40 + 3, 2 ** 33 + 8, 123456789),
                                          (0xDEADBEEFCAFE, 65528, 2 ** 32 + 7)])
def test_swap_uniform_known_answers(seed, chain, n):
    from oracle import ladder_oracle as co
    x, y, _, _ = philox4x32_7([chain & 0xFFFFFFFF, chain >> 32, n & 0xFFFFFFFF, 0xFFFFFFFF],
                              [seed & 0xFFFFFFFF, seed >> 32])
    K = (y << 20) | (x >> 12)
    assert co.swap_uniform(seed, chain, n) == (K + 0.5) * 2.0 ** -52


def test_swap_uniform_is_not_a_step_draw():
    """Slot 0xFFFFFFFF is no step slot: the swap uniform differs from the radius uniform of every step slot."""
    from oracle import ladder_oracle as co
    for q in range(16):
        x, y, _, _ = philox4x32_7([9, 0, 4, q], [1, 0])
        assert co.swap_uniform(1, 9, 4) != (((y << 20) | (x >> 12)) + 0.5) * 2.0 ** -52


def test_two_rung_x2_ladder_samples_each_temperature():
    """E = x^2 at T: variance T/2.  4,096 independent ladders, one sample per rung from each."""
    from oracle import ladder_oracle as co
    temps, n_lad = [0.5, 2.0], 4096
    xs = np.empty((n_lad, 2))
    for i in range(n_lad):
        lad = co.CLadder(1, 0, "x2", temps, swap_every=1, x0=np.zeros(1), chain0=2 * i, sampling_width=0.5)
        lad.run(100, 10, seed=11)
        xs[i] = lad.x[:, 0]
    for r, t in enumerate(temps):
        var = np.mean(xs[:, r] ** 2)                  # the mean is 0 by symmetry
        se = np.std(xs[:, r] ** 2) / np.sqrt(n_lad)
        assert abs(var - t / 2) < 5 * se, (r, var, t / 2, se)


@pytest.mark.parametrize("R,every,blocks", [(2, 1, 30), (4, 3, 31), (8, 2, 40), (8, 5, 9)])
def test_swap_attempts_follow_the_even_odd_schedule(R, every, blocks):
    from oracle import ladder_oracle as co
    from metropolisengine_b200.engine import MetropolisEngine
    lad = co.CLadder(2, 0, "xy_well", np.geomspace(0.1, 1.0, R), consts=[1.0], swap_every=every, x0=np.zeros(2))
    lad.run(blocks, 3, seed=2)
    n_last = lad.n_measure.value
    rounds = [k for k in range(1, n_last // every + 1) if k * every >= 2]      # counters n = 2 .. n_last
    want = [sum(1 for k in rounds if k % 2 == r % 2) for r in range(R - 1)]
    assert list(lad.swap_att[:R - 1]) == want
    assert lad.swap_att[R - 1] == 0 and lad.swap_acc[R - 1] == 0

    class Probe:                                        # the engine's count from the counter alone
        _ladder, _swap_every, measure_step_counter = np.zeros(R), every, n_last
    assert list(MetropolisEngine._swap_attempts(Probe())) == want
    assert sorted(lad.walker) == list(range(R))          # a permutation of the labels
