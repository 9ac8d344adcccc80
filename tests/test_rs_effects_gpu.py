"""Global effect chains of Rust-API engines on the GPU (gooey_rs_batch_add_effect, rs_chain_kernel) against the oracle's
RustEngine: every kind alone, the examples/bounce.rs chain, batches mixing chains with limiter-only engines, effect
state across bounces, refusals, device-resident output, and the 4096-engine workload of tools/rs_effects_bench.py."""
import ctypes as c
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from libgooey_b200 import bounce as B
from rs_effects_oracle import ARGS, EXAMPLE_CHAIN, RustOracle

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import rs_effects_bench as W  # noqa: E402

pytestmark = pytest.mark.gpu
TOL = 1e-5
SR = 44100.0
BAR = 88200


def add(batch, i, eid, args):
    a = np.array(list(args) or [0.0], np.float32)
    return B._L().gooey_rs_batch_add_effect(batch._h, i, eid, a.ctypes.data, len(args))


def setup(batch, i, seed=3, master=None):
    insts, seqs, m = W.engine_spec(i, seed)
    e = batch[i]
    for name, inst in insts:
        e.add_instrument(name, inst)
    for name, en, ve in seqs:
        e.add_sequencer(B.Sequencer.with_velocity_pattern(120.0, SR, list(zip(en.tolist(), ve.tolist())), name))
    e.set_master_gain(m if master is None else master)
    return insts, seqs, (m if master is None else master)


def oracle(i, limiter, effects, seed=3, bounces=1, samples=BAR):
    insts, seqs, m = W.engine_spec(i, seed)
    o = RustOracle(insts, seqs, master=m, limiter=limiter, effects=effects)
    out = [o.bounce(samples) for _ in range(bounces)]
    o.close()
    return out


def scaled(eid, k):
    """Engine k's constructor arguments of kind eid: ARGS varied per engine (timing and integer-like args kept)."""
    if eid == 1:
        t, bpm, fb, mix, cut = ARGS[1]
        return ((t + k) % 9, bpm + 3 * k, fb * (1 - 0.05 * k), mix, cut - 300 * k)
    return tuple(a * (1.0 - 0.04 * k) for a in ARGS[eid])


@pytest.mark.parametrize("eid", list(range(10)))
def test_each_kind_alone_matches_the_oracle(eid):
    n = 8
    batch = B.EngineBatch(n, SR)
    for k in range(n):
        setup(batch, k)
        batch[k].clear_global_effects()
        assert add(batch, k, eid, scaled(eid, k)) == 0
    got = batch.bounce(B.BounceLength.Bars(1))
    batch.close()
    for k in range(n):
        want = oracle(k, False, [(eid, scaled(eid, k))])[0]
        err = np.abs(got[k] - want).max()
        assert np.abs(want).max() > 0.01
        assert err <= TOL, (k, err)


@pytest.mark.parametrize("keep_default", [True, False])
def test_bounce_rs_example_chain_matches_the_oracle(keep_default):
    n = 32
    batch = B.EngineBatch(n, SR)
    for k in range(n):
        setup(batch, k)
        e = batch[k]
        if not keep_default:
            e.clear_global_effects()
        e.add_global_effect(B.TubeSaturation(SR, 0.3, 0.4, 0.5))
        e.add_global_effect(B.DelayEffect(SR, 3, 128.0, 0.35, 0.2, 8000.0))
        e.add_global_effect(B.TubeCompressor(SR, -12.0, 4.0, 10.0, 100.0, 0.6))
        e.add_global_effect(B.SoftLimiter(0.95))
    got = batch.bounce(B.BounceLength.Bars(1))
    batch.close()
    for k in range(n):
        want = oracle(k, keep_default, EXAMPLE_CHAIN)[0]
        assert np.abs(want).max() > 0.01
        assert np.abs(got[k] - want).max() <= TOL, k


LIMITER_ONLY = [[], None, [0.5], [0.8, 0.6], [0.9, 0.9, 0.7, 0.5]]   # None = the default chain


def test_limiter_only_engines_are_untouched_by_effect_engines_in_the_batch():
    def make(with_fx):
        n = len(LIMITER_ONLY) + (3 if with_fx else 0)
        batch = B.EngineBatch(n, SR)
        for k, lims in enumerate(LIMITER_ONLY):
            setup(batch, k)
            if lims is not None:
                batch[k].clear_global_effects()
                for th in lims:
                    batch[k].add_global_effect(B.SoftLimiter(th))
        if with_fx:
            for k, chain in zip(range(len(LIMITER_ONLY), n), ([(9, ARGS[9])], [(5, (0.7,)), (1, ARGS[1])], [(5, (0.9,))] * 5)):
                setup(batch, k)
                for eid, args in chain:
                    assert add(batch, k, eid, args) == 0
        return batch
    a, b = make(True), make(False)
    got_a = [a.bounce(B.BounceLength.Bars(1)) for _ in range(2)]
    got_b = [b.bounce(B.BounceLength.Bars(1)) for _ in range(2)]
    m = len(LIMITER_ONLY)
    for x, y in zip(got_a, got_b):
        assert np.array_equal(x[:m], y)
    # the effect engines against the oracle, second bounce included (five limiters: more than rs_mix_kernel takes)
    for k, chain in zip(range(m, m + 3), ([(9, ARGS[9])], [(5, (0.7,)), (1, ARGS[1])], [(5, (0.9,))] * 5)):
        want = oracle(k, True, chain, bounces=2)
        for r in range(2):
            assert np.abs(got_a[r][k] - want[r]).max() <= TOL, (k, r)
    for k, lims in enumerate(LIMITER_ONLY):
        want = oracle(k, lims is None, [(5, (th,)) for th in (lims or [])])[0]
        assert np.abs(got_a[0][k] - want).max() <= TOL, k
    a.close(); b.close()


def test_state_carries_across_bounces_clear_starts_fresh_and_bpm_leaves_the_delay_alone():
    chain = [(9, ARGS[9]), (1, ARGS[1])]
    batch = B.EngineBatch(3, SR)
    for k in range(3):
        setup(batch, k)
        batch[k].clear_global_effects()
        for eid, args in chain:
            assert add(batch, k, eid, args) == 0
    L = B._L()
    n = BAR // 2
    g1 = batch.bounce(B.BounceLength.Samples(n))
    # engine 1: cleared and rebuilt (fresh lines); engine 2: new tempo, which the delay does not see
    batch[1].clear_global_effects()
    for eid, args in chain:
        assert add(batch, 1, eid, args) == 0
    assert L.gooey_rs_batch_set_bpm(batch._h, 2, c.c_float(90.0)) == 0
    g2 = batch.bounce(B.BounceLength.Samples(n))
    batch.close()
    for k in range(3):
        insts, seqs, m = W.engine_spec(k, 3)
        o = RustOracle(insts, seqs, master=m, limiter=False, effects=chain)
        w1 = o.bounce(n)
        if k == 1:
            o.clear()
            for eid, args in chain:
                o.add_effect(eid, args)
        if k == 2:
            o.set_bpm(90.0)
        w2 = o.bounce(n)
        o.close()
        assert np.abs(g1[k] - w1).max() <= TOL, k
        assert np.abs(g2[k] - w2).max() <= TOL, k
    fresh = oracle(0, False, chain, samples=n)[0]
    assert np.abs(g2[0] - fresh).max() > 1e-3        # engine 0 carries its tails


def test_refusals_leave_the_chain_unchanged():
    batch = B.EngineBatch(2, SR)
    setup(batch, 0)
    L = B._L()
    L.gooey_b200_last_error.restype = c.c_char_p
    INVALID = -1   # GOOEY_E_INVALID
    one = np.array([0.5, 0.5, 0.5, 0.5, 0.5], np.float32)
    bad = [lambda: L.gooey_rs_batch_add_effect(batch._h, 0, 10, one.ctypes.data, 0),
           lambda: L.gooey_rs_batch_add_effect(batch._h, 0, 0xFFFFFFFF, one.ctypes.data, 1),
           lambda: L.gooey_rs_batch_add_effect(batch._h, 0, 9, one.ctypes.data, 2),
           lambda: L.gooey_rs_batch_add_effect(batch._h, 0, 9, None, 3),
           lambda: L.gooey_rs_batch_add_effect(batch._h, 2, 9, one.ctypes.data, 3)]
    codes = []
    for f in bad:
        codes.append(f())
        assert L.gooey_b200_last_error()
    # the default limiter + 7 more fill the chain; the 9th is refused
    for _ in range(7):
        assert add(batch, 0, 5, (0.9,)) == 0
    codes.append(add(batch, 0, 5, (0.9,)))
    assert L.gooey_b200_last_error()
    codes.append(L.gooey_rs_batch_add_limiter(batch._h, 0, c.c_float(0.9)))
    assert codes == [INVALID] * len(codes)
    got = batch.bounce(B.BounceLength.Bars(1))[0]
    batch.close()
    want = oracle(0, True, [(5, (0.9,))] * 7)[0]
    assert np.abs(got - want).max() <= TOL


def test_device_bounce_with_a_wide_stride_gives_the_host_rows():
    torch = pytest.importorskip("torch")
    chain = [(2, ARGS[2]), (6, ARGS[6]), (5, (0.8,))]
    outs = []
    for device in (False, True):
        batch = B.EngineBatch(40, SR)
        for k in range(40):
            setup(batch, k)
            for eid, args in chain:
                assert add(batch, k, eid, args) == 0
        n = 10001
        if device:
            stride = 10240 + 3
            buf = torch.full((40, stride), 7.0, dtype=torch.float32, device="cuda")
            assert B._L().gooey_rs_batch_bounce_device(batch._h, n, c.c_void_p(buf.data_ptr()), stride) == 0
            torch.cuda.synchronize()
            h = buf.cpu().numpy()
            assert (h[:, n:] == 7.0).all()
            outs.append(h[:, :n])
        else:
            outs.append(batch.bounce(B.BounceLength.Samples(n)))
        batch.close()
    assert np.array_equal(outs[0], outs[1])


def test_bench_workload_4096_engines_every_64th_matches_the_oracle():
    n = 4096
    for chain in ("b_bounce_rs_example", "c_plate_delay_limiter"):
        batch = W.build_batch(n, chain, seed=7)
        got = batch.bounce(B.BounceLength.Bars(1))
        batch.close()
        keep, effects = W.CHAINS[chain]

        def one(i):
            insts, seqs, m = W.engine_spec(i, 7)
            o = RustOracle(insts, seqs, master=m, limiter=keep, effects=effects)
            w = o.bounce(BAR)
            o.close()
            return i, w
        with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
            for i, w in ex.map(one, range(0, n, 64)):
                assert np.abs(got[i] - w).max() <= TOL, (chain, i)
