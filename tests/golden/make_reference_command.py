"""Extracts the container `command:` and `image:` of the reference Deployment
(cuda-test-deployment.yaml:18-19) into tests/golden/reference_command.json.

The reference is not part of this repository, so the parsed values are committed as a
fixture; tests/test_image_layout.py drives the runtime layout with that command and checks
that parse() reads the fixture back from a Deployment carrying it.

    python tests/golden/make_reference_command.py <reference checkout>
"""
import json
import os
import sys

import yaml

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_command.json")


def parse(path: str) -> dict:
    doc = yaml.safe_load(open(path))
    c = doc["spec"]["template"]["spec"]["containers"][0]
    return {"source": "cuda-test-deployment.yaml:18-19", "container": c["name"], "image": c["image"], "command": c["command"],
            "gpu_limit": c["resources"]["limits"]["nvidia.com/gpu"]}


if __name__ == "__main__":
    json.dump(parse(os.path.join(sys.argv[1], "cuda-test-deployment.yaml")), open(OUT, "w"), indent=1)
    print(open(OUT).read())
