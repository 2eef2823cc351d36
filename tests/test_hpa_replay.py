"""The control-loop arithmetic of the (unchanged) manifests, restated offline."""
import os

import pytest

from conftest import ROOT
from k8s_gpu_hpa_b200 import hpa_replay as hr


def test_constants_match_the_reference_manifests():
    """The values the reference's manifests set, as extracted by tests/golden/make_reference_manifests.py."""
    import json

    ref = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_manifests.json")))
    assert hr.HPA_TARGET == ref["hpa_target_value"]
    assert (hr.HPA_MIN, hr.HPA_MAX) == (ref["hpa_min_replicas"], ref["hpa_max_replicas"])
    assert ref["hpa_metric"] == hr.cuda_test_gpu_avg.__name__
    assert hr.DCGM_INTERVAL_S * 1000 == ref["dcgm_collect_interval_ms"]
    assert f"{hr.SCRAPE_INTERVAL_S:g}s" == ref["scrape_interval"]


def test_recording_rule_max_by_pod_then_avg_over_labelled_pods():
    S = hr.Sample
    dcgm = [S("n0", "cuda-test-a", "default", 12.0, "0"), S("n0", "cuda-test-a", "default", 30.0, "1"),   # 2 GPUs, one pod
            S("n1", "cuda-test-b", "default", 10.0), S("n1", "other-pod", "default", 99.0)]
    labels = {"cuda-test-a": "cuda-test", "cuda-test-b": "cuda-test", "other-pod": "something-else"}
    assert hr.cuda_test_gpu_avg(dcgm, labels) == pytest.approx((30.0 + 10.0) / 2)
    assert hr.cuda_test_gpu_avg([S("n1", "other-pod", "default", 99.0)], labels) is None


@pytest.mark.parametrize("current,metric,want", [
    (1, 4.0, 1), (1, 5.0, 1), (1, 5.4, 1),       # inside the 10 % tolerance band
    (1, 5.6, 2), (1, 9.9, 2), (1, 10.1, 3), (1, 99.0, 3),
    (2, 5.6, 3), (3, 50.0, 3),                   # maxReplicas clamp
    (3, 1.0, 1), (2, 2.4, 1), (3, 3.0, 2),       # scale-down ("if the usage drops low enough")
    (1, None, 1), (1, 0.0, 1),
])
def test_hpa_decision(current, metric, want):
    assert hr.hpa_desired_replicas(current, metric) == want


def test_replay_reference_shape_vs_sustained_loop():
    # the reference's duty cycle (process churn) sits under the threshold; a sustained
    # in-process loop crosses it and the overshoot the README warns about appears
    idle = {"cuda-test-0": [(t, 3.0) for t in range(0, 120)]}
    r = hr.Replay()
    assert all(rep == 1 for _, _, rep in r.run(idle, 120))
    busy = {f"cuda-test-{i}": [(t, 97.0) for t in range(0, 120)] for i in range(3)}
    ev = r.run(busy, 120)
    assert ev[0][2] == 3 or ev[1][2] == 3                       # jumps straight to maxReplicas
    assert hr.would_scale_up(6.0) and not hr.would_scale_up(5.2)


@pytest.mark.parametrize("rel", ["r01/aa_hpa_trigger_replay.jsonl", "r02/e_hpa_trigger_replay.jsonl"])
def test_recorded_gpu_run_replays_to_the_same_decisions(rel):
    """profiles/r0x/*_hpa_trigger_replay.jsonl: NVML utilisation measured on a B200 while the
    load generator ran at several duty cycles; the offline rule + HPA must agree with it."""
    import json

    path = os.path.join(ROOT, "profiles", *rel.split("/"))
    if not os.path.exists(path):
        pytest.skip("recorded run not present")
    rows = [json.loads(l) for l in open(path)]
    assert len(rows) >= 5
    for r in rows:
        want_up = r["nvml_util_mean"] > hr.HPA_TARGET * (1 + hr.HPA_TOLERANCE)
        assert hr.would_scale_up(r["nvml_util_mean"]) == want_up == r["steady_state_would_scale_up"]
        final_replicas = r["replay_events_t_metric_replicas"][-1][2]
        assert (final_replicas > 1) == want_up
        if isinstance(r["target_util"], (int, float)):
            assert abs(r["nvml_util_mean"] - r["target_util"]) <= max(1.0, 0.1 * r["target_util"])   # controller accuracy


def test_scale_down_waits_for_the_stabilization_window():
    """kube-controller-manager's default 5-minute downscale stabilization: after the load stops the
    replicas stay up until every recommendation of the last 300 s is lower; scale-ups are immediate."""
    trace = {f"cuda-test-{i}": [(t, 97.0 if t < 60 else 1.0) for t in range(0, 600)] for i in range(3)}
    ev = hr.Replay().run(trace, 600)
    up = [t for t, _, r in ev if r == 3]
    assert up and up[0] <= 30                                       # straight to maxReplicas
    first_down = min(t for t, _, r in ev if t > 60 and r < 3)
    assert 60 + 300 <= first_down <= 60 + 300 + 3 * hr.HPA_SYNC_S   # not before the window has passed
    assert ev[-1][2] == 1
    # without the window the same trace drops at the next sync
    ev0 = hr.Replay(downscale_stabilization_s=0.0).run(trace, 600)
    assert min(t for t, _, r in ev0 if t > 60 and r < 3) <= 60 + hr.DCGM_INTERVAL_S + 2 * hr.HPA_SYNC_S
