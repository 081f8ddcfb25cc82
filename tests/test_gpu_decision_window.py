"""The throughput build's Metropolis decision (me_device.cuh, Rng::accept_window / finish_step) compares FP32(dE) with an
FP32 window around the threshold -T ln u and falls back to the exact FP64 test inside it.  Every decision must equal the
exact test, so a fast ensemble must follow the C oracle (exact FP64 decisions on the same Philox streams) chain by chain:
identical acceptance counts, state within the throughput build's 2e-9.

2,048 chains x 2,000 steps put roughly 80 decisions inside the window per case (probability ~2e-5 per step), plus the
wide windows of accept words below 2^18.  T = 0 checks the window that sends an FP32 dE of +-0 to the exact test; the
x^2 shape (D = 1) checks both steps of the Philox call that two consecutive steps share."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SHAPES = [
    ("xy_well", 2, [1.0]),
    ("x2", 1, []),
]


@pytest.mark.parametrize("temp", [0.0, 1e-3, 0.1, 10.0])
@pytest.mark.parametrize("bname,n_r,consts", SHAPES)
def test_fast_decisions_equal_exact_test_chain_by_chain(bname, n_r, consts, temp):
    import metropolisengine_b200 as me
    from oracle import c_oracle as co
    n, M, K, seed = 2048, 200, 10, 77
    x0 = np.full(n_r, 0.5)
    eng = me.MetropolisEngine(me.BuiltinEnergy(bname, *consts), initial_real_params=x0, n_chains=n, seed=seed,
                              temp=temp)
    eng.run(M, K)
    eng.check_status()
    st = eng.state.cpu().numpy()
    lay = eng._lay
    words = lay.WORDS - 2                              # everything but the acceptance count and the status word
    bad_nacc, bad_state = [], []
    for ch in range(n):
        o = co.CChain(n_r, 0, bname, consts=consts, temp=temp, x0=x0)
        acc, _ = o.run(M, K, True, seed=seed, chain_id=ch)
        if st[lay.NACC, ch] != acc.sum():
            bad_nacc.append((ch, st[lay.NACC, ch], int(acc.sum())))
        ref = o.state[:words]
        scale = max(np.max(np.abs(ref)), 1e-300)
        if not np.all(np.abs(st[:words, ch] - ref) <= 2e-9 * np.maximum(np.abs(ref), scale)):
            bad_state.append(ch)
    assert not bad_nacc, bad_nacc[:10]
    assert not bad_state, bad_state[:10]
    assert np.all(st[lay.STATUS] == 0)
