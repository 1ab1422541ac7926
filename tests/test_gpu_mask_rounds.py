"""Rounds of the mask run that take zone-unpinned nodes (DESIGN.md section 4, "Rounds"): a zone-spread class with max skew 1
places one pod in each admissible zone per round, and unpinned open nodes that come first in the order are pinned inside
the round to the lowest open zone, as the one-pod step does. These inputs put such nodes in front of the spread classes;
every result must be the oracle's (or, at sizes the oracle is too slow for, the per-pod loop's) bit for bit."""
import numpy as np
import pytest

import fixtures as fx

pytestmark = pytest.mark.gpu

MODES = ("KSCHED_NO_LEVELWARP", "KSCHED_NO_MASKRUN", "KSCHED_NO_LEVELRUN", "KSCHED_NO_CLASSRUN")


def _match_oracle(pkg, oracle, problem):
    got = pkg.Scheduler(problem).solve()
    want = pkg.Result()
    assert oracle.solve(problem, want) == 0, want.error
    assert np.array_equal(got.assign, want.assign)
    assert got.num_new_nodes == want.num_new_nodes
    assert got.digest() == want.digest()
    return got


@pytest.mark.parametrize("seed", [1, 2, 5, 13, 29])
def test_c4_samples_match_oracle(pkg, oracle, seed):
    _match_oracle(pkg, oracle, pkg.Problem.synth(4, 2500 + 100 * (seed % 6), 1000, seed, 0))


@pytest.mark.parametrize("pods,seed", [(20000, 3), (35000, 17), (50000, 42)])
def test_c4_mask_run_matches_per_pod_loop(pkg, monkeypatch, pods, seed):
    """The per-pod loop (KSCHED_NO_MASKRUN) places one pod at a time and is the reference the rounds must reproduce."""
    rs = pkg.ResidentSolve(pkg.Problem.synth(4, pods, 1000, seed, 0))
    rs.set_count_visited(False)
    rs.load()
    out = {}
    for off in ("", "KSCHED_NO_MASKRUN"):
        for v in MODES:
            monkeypatch.delenv(v, raising=False)
        if off:
            monkeypatch.setenv(off, "1")
        rs.run()
        res = rs.download()
        out[off or "mask run"] = (int(res.digest()), int(res.num_new_nodes), int((res.assign >= 0).sum()))
    for v in MODES:
        monkeypatch.delenv(v, raising=False)
    assert out["mask run"] == out["KSCHED_NO_MASKRUN"], out


def _unpinned_first(instance_types=None, n_anti=7, n_spread=40):
    """A hostname anti-affinity deployment opens one node per pod, none of them pinned to a zone and each with room for
    four more pods; a max-skew-1 zone spread deployment with smaller pods follows and meets those nodes first."""
    anti = {"app": "anti"}
    pods = [fx.pod({"cpu": "1"}, labels=anti,
                   podAntiAffinity={"required": [fx.affinity_term(fx.HOSTNAME, anti)]})
            for _ in range(n_anti)]
    spread = {"app": "spread"}
    pods += [fx.pod({"cpu": "500m"}, labels=spread, topologySpreadConstraints=[fx.spread(fx.ZONE, spread)]) for _ in range(n_spread)]
    return fx.problem(pods, instance_types=instance_types)


def test_unpinned_nodes_before_zone_spread(pkg, oracle):
    _match_oracle(pkg, oracle, pkg.Problem.from_dict(_unpinned_first()))


@pytest.mark.parametrize("n_anti", [2, 4, 11])
def test_unpinned_node_counts(pkg, oracle, n_anti):
    _match_oracle(pkg, oracle, pkg.Problem.from_dict(_unpinned_first(n_anti=n_anti, n_spread=31)))


def test_unpinned_pin_not_neutral(pkg, oracle):
    """One instance type is offered in two zones only: pinning a node to the third one drops an option, which the round
    cannot represent, so that pod takes the one-pod step and the generic step behind it."""
    its = [fx.instance_type("default-instance-type"),
           fx.instance_type("two-zone-type", {"cpu": "8", "memory": "8Gi"},
                            offerings=[{"capacityType": "on-demand", "zone": z, "price": 0.5, "available": True} for z in fx.ZONES[:2]])]
    _match_oracle(pkg, oracle, pkg.Problem.from_dict(_unpinned_first(instance_types=its)))
