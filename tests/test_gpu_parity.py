"""GPU parity: the CUDA path (through the C ABI of libserfsim.so) against the CPU oracle, bit for bit.

Compared on the same seeded inputs: the raw 32-byte member records of every slot, the Lamport clock
of every node, the memberlist state/incarnation vectors, the convergence step count and EVERY field
of EVERY row of the per-tick trace (packets, edge-updates, messages, changed, pending, events,
suspects, state hash).  Integer work: the bar is exact equality.
"""
import numpy as np
import pytest

from oracle_lib import oracle_sim
from serf_b200 import GossipSim, MemberStatus, scenarios

pytestmark = pytest.mark.gpu


def gpu_sim(n, slots=1, **kw):
    return GossipSim(n, slots, **kw)


def assert_same(g, o, slots):
    sg, so = g.stats(), o.stats()
    assert sg == so, (sg, so)
    n = sg["tick"]
    tg, to = g.tick_trace(0, n), o.tick_trace(0, n)
    for f in tg.dtype.names:
        bad = np.nonzero(tg[f] != to[f])[0]
        assert bad.size == 0, f"trace field {f} first differs at tick {bad[0]}: gpu {tg[f][bad[0]]} oracle {to[f][bad[0]]}"
    assert (g.lamport_time() == o.lamport_time()).all()
    assert (g.lamport_time_u32() == o.lamport_time()).all()
    for s in range(slots):
        rg, ro = g.records(s), o.records(s)
        bad = np.nonzero(rg != ro)[0]
        assert bad.size == 0, f"slot {s}: record of node {bad[0]} differs: gpu {rg[bad[0]]} oracle {ro[bad[0]]}"
        assert (g.member_status(s) == o.member_status(s)).all()
        assert (g.status_ltime(s) == o.status_ltime(s)).all()
        assert (g.status_ltime_u32(s) == o.status_ltime(s)).all()                 # compact getters: same values, half the bytes
        assert (g.incarnation(s) == o.incarnation(s)).all()
        assert (g.ml_state(s) == o.ml_state(s)).all()
    assert g.state_hash() == o.state_hash()


def run_both(sc, **cfg):
    g, o = sc.build(gpu_sim, trace=1, **cfg), sc.build(oracle_sim, trace=1, **cfg)
    tg, okg = g.run_until_converged(sc.max_ticks)
    to, oko = o.run_until_converged(sc.max_ticks)
    assert (tg, okg) == (to, oko), f"convergence step count differs: gpu {(tg, okg)} oracle {(to, oko)}"
    assert_same(g, o, sc.slots)
    # production mode (trace = 0): idle tiles are skipped and no per-tick hash is computed; everything
    # else — every other trace field, the records, the clocks, the final state hash — must still be equal
    f = sc.build(gpu_sim, trace=0, **cfg)
    tf, okf = f.run_until_converged(sc.max_ticks)
    assert (tf, okf) == (to, oko)
    n = o.stats()["tick"]
    trf, tro = f.tick_trace(0, n), o.tick_trace(0, n)
    for name in trf.dtype.names:
        if name != "hash":
            bad = np.nonzero(trf[name] != tro[name])[0]
            assert bad.size == 0, f"trace=0: field {name} first differs at tick {bad[0]}"
    assert f.state_hash() == o.state_hash() and f.stats() == o.stats()
    for s in range(sc.slots):
        assert (f.records(s) == o.records(s)).all()
    assert (f.lamport_time() == o.lamport_time()).all()
    return g, o, tg


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_config0_full_mesh_256(seed):
    g, o, ticks = run_both(scenarios.full_mesh_leave(256, 3, seed))
    assert (g.member_status(0)[1:] == MemberStatus.LEFT).all()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_config1_random_graph_100k(seed):
    g, o, ticks = run_both(scenarios.random_graph_leave(100_000, 16, 3, seed))
    assert (g.member_status(0)[1:] != MemberStatus.LEFT).sum() <= 3 and ticks < 100     # a random digraph may strand a node or two


def test_random_graph_fanout4_ragged_tail():
    run_both(scenarios.random_graph_leave(60_001, 12, 4, seed=5))          # single slot, last tile partly filled


def test_random_graph_multi_slot_fanout4():
    run_both(scenarios.random_graph_leave(60_000, 16, 4, seed=5, slots=4))


def test_failure_detection_random_graph():
    sc = scenarios.random_graph_fail(20_000, 16, 3, seed=2)
    g, o, ticks = run_both(sc, suspicion_mult=2, suspicion_max_timeout_mult=2, probe_interval_ticks=2)
    st = g.member_status(0)
    assert (np.delete(st, 5) == MemberStatus.FAILED).all()


def test_failure_detection_single_subject():
    sc = scenarios.random_graph_fail(20_000, 16, 3, seed=2)
    sc.slots, sc.subjects, sc.ops = 1, sc.subjects[:1], [op for op in sc.ops if op[2] == int(sc.subjects[0])]
    run_both(sc, suspicion_mult=2, suspicion_max_timeout_mult=2, probe_interval_ticks=2)


def test_failure_detection_lifeguard_confirmations():
    sc = scenarios.random_graph_fail(5_000, 24, 3, seed=4)
    run_both(sc, suspicion_mult=4, suspicion_max_timeout_mult=3, probe_interval_ticks=1, gossip_interval_ms=1000)


def test_config2_small_world_churn():
    sc = scenarios.small_world_churn(40_000, 16, 0.1, 0.05, slots=8, window=60, seed=3)
    run_both(sc, suspicion_mult=2, suspicion_max_timeout_mult=2, probe_interval_ticks=2)


@pytest.mark.parametrize("pp", [7, 16])
def test_push_pull_anti_entropy(pp):
    from serf_b200 import small_world_graph
    from serf_b200.scenarios import Scenario
    from serf_b200 import Op
    n = 20_000
    sc = Scenario("pushpull", n, 3, small_world_graph(n, 4, 0.05, 5), [7, 900, 15000],
                  [(0, Op.LEAVE, 7, 0), (3, Op.FAIL, 900, 0), (40, Op.FORCE_LEAVE, 11, 1), (5, Op.JOIN, 15000, 0)],
                  dict(fanout=2, retransmit_mult=1, seed=5, push_pull_interval_ticks=pp, probe_interval_ticks=2, suspicion_mult=2, suspicion_max_timeout_mult=2), max_ticks=3000)
    g, o, ticks = run_both(sc)
    assert (ticks + 1) % pp == 0


@pytest.mark.parametrize("seed", range(40))
def test_fuzz(seed):
    sc = scenarios.fuzz(seed)
    sc.max_ticks = 1500
    run_both(sc)


@pytest.mark.parametrize("seed", range(12))
def test_fuzz_single_slot(seed):
    sc = scenarios.fuzz(seed, slots=1)
    sc.max_ticks = 1500
    run_both(sc)


def test_remove_failed_node_prune_reference_scenario():
    """serf_remove_failed_node_prune (serf/base/tests/serf/remove.rs:95-165) and the same on a 20 K-node random graph: after the
    pruning force-leave no survivor lists the failed node any more."""
    for n in (3, 40, 20_000):
        g, o, ticks = run_both(scenarios.remove_failed_node_prune(n, at=40 if n < 1000 else 120))
        st = g.member_status(0)
        assert (np.delete(st, 1) != MemberStatus.NONE).sum() <= (0 if n < 1000 else 3)


@pytest.mark.parametrize("seed", range(24))
def test_fuzz_prune(seed):
    sc = scenarios.fuzz_prune(seed)
    sc.max_ticks = 1500
    run_both(sc)


def test_stepwise_equals_batched_and_inject_midway():
    sc = scenarios.random_graph_leave(30_000, 16, 3, seed=8, slots=2)
    g, o = sc.build(gpu_sim, trace=1), sc.build(oracle_sim, trace=1)
    for _ in range(6):
        g.step(1); o.step(1)
    g.remove_failed_node(77, 1, tick=9); o.remove_failed_node(77, 1, tick=9)
    g.step(7); o.step(7)
    assert_same(g, o, 2)
    tg, to = g.run_until_converged(500), o.run_until_converged(500)
    assert tg == to
    assert_same(g, o, 2)


def test_reset_reproduces():
    sc = scenarios.random_graph_leave(50_000, 16, 3, seed=4)
    g = sc.build(gpu_sim, trace=1)
    t1, _ = g.run_until_converged(500)
    h1, tr1 = g.state_hash(), g.tick_trace()
    g.reset(4)
    sc.schedule(g)
    t2, _ = g.run_until_converged(500)
    assert (t1, h1) == (t2, g.state_hash()) and (tr1 == g.tick_trace()).all()


def test_event_callback_reports_agreed_transitions():
    sc = scenarios.full_mesh_leave(256, 3, 1)
    g = sc.build(gpu_sim)
    seen = []
    g.set_event_callback(lambda tick, ty, ids: seen.append((ty, tuple(ids))))
    g.run_until_converged(500)
    assert (1, (0,)) in seen            # MemberEventType::Leave for subject 0


def others_mask(status, subj):
    m = status != MemberStatus.LEFT
    m[subj] = False
    return m


# ---- full-size properties (no oracle at this size): BASELINE configs[3] shape on one GPU ----------
def test_full_size_10m_properties():
    sc = scenarios.dissemination_storm(10_000_000, 16, 4, slots=1, seed=1)
    g = sc.build(gpu_sim, trace=1)
    ticks, ok = g.run_until_converged(400)
    assert ok
    st = g.stats()
    h1, tr1 = g.state_hash(), g.tick_trace()
    status = g.member_status(0)
    subj = int(sc.subjects[0])
    assert status[subj] == MemberStatus.LEAVING
    # a random digraph with Poisson(16) in-degree leaves O(1) of 10 M nodes unreachable (in-degree 0): they stay Alive
    others = np.delete(status, subj)
    missed = int((others != MemberStatus.LEFT).sum())
    assert missed <= 8 and set(np.unique(others)) <= {MemberStatus.ALIVE, MemberStatus.LEAVING, MemberStatus.LEFT, MemberStatus.FAILED}
    lt = g.status_ltime(0)
    assert ((lt == 2) | (others_mask(status, subj) & (lt == 1))).all()
    # every node that accepted an entry forwards it exactly retransmit_limit (32) times
    reached_intent = int((lt == 2).sum())
    reached_left = int((g.ml_state(0) == 3).sum())
    assert st["messages"] == 32 * (reached_intent + reached_left) and st["intent_queue"] == 0 and st["pending"] == 0
    assert tr1["hash"][-1] == h1
    # idempotence / determinism: same seed → same trace; extra ticks on a quiescent cluster change nothing
    g.step(3)
    assert g.state_hash() == h1
    g.reset(1); sc.schedule(g)
    t2, _ = g.run_until_converged(400)
    assert t2 == ticks and g.state_hash() == h1 and (g.tick_trace() == tr1).all()
