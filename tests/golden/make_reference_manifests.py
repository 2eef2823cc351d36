"""Extracts the control-loop constants of the reference's manifests into
tests/golden/reference_manifests.json: the HPA's replica bounds, metric and target
(cuda-test-hpa.yaml), dcgm-exporter's collection interval (dcgm-exporter.yaml) and the GPU
job's Prometheus scrape interval (kube-prometheus-stack-values.yaml).

The reference is not part of this repository, so the extracted values are committed as a
fixture; tests/test_hpa_replay.py checks the constants of hpa_replay.py against it.

    python tests/golden/make_reference_manifests.py <reference checkout>
"""
import json
import os
import sys

import yaml

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_manifests.json")


def parse(ref: str) -> dict:
    def load(name):
        return list(yaml.safe_load_all(open(os.path.join(ref, name))))

    hpa = load("cuda-test-hpa.yaml")[0]["spec"]
    obj = hpa["metrics"][0]["object"]
    dcgm = [d for d in load("dcgm-exporter.yaml") if d and d.get("kind") == "DaemonSet"][0]
    args = dcgm["spec"]["template"]["spec"]["containers"][0]["args"]
    jobs = load("kube-prometheus-stack-values.yaml")[0]["prometheus"]["prometheusSpec"]["additionalScrapeConfigs"]
    gpu_job = [j for j in jobs if j["job_name"] == "gpu-metrics"][0]
    return {"source": ["cuda-test-hpa.yaml", "dcgm-exporter.yaml", "kube-prometheus-stack-values.yaml"],
            "hpa_min_replicas": hpa["minReplicas"], "hpa_max_replicas": hpa["maxReplicas"],
            "hpa_metric": obj["metricName"], "hpa_target_value": obj["targetValue"],
            "dcgm_collect_interval_ms": int(args[args.index("-c") + 1]),
            "scrape_interval": gpu_job["scrape_interval"]}


if __name__ == "__main__":
    json.dump(parse(sys.argv[1]), open(OUT, "w"), indent=1)
    print(open(OUT).read())
