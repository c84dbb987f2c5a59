"""Generates tests/golden/fetch_model_facts.json, the numbers tests/test_model_compiler.py checks the committed model blobs against,
from the reference's MJCF assets (B200SIM_REFERENCE_ASSETS, see gymnasium_robotics_b200/models.py); the assets themselves are not
redistributed, so the tests read this file instead:
  - blob_sha256: SHA-256 of a fresh compile of every MODEL_SOURCES entry (what the committed blobs must be);
  - fetch_robot_xml: per-body subtree masses summed from the <inertial mass=...> entries of fetch/robot.xml, read with ElementTree
    (every link there has an explicit <inertial>), and the <inertial pos> of robot0:gripper_link;
  - fetch_pick_and_place_mjcf: the number of MJCF bodies (world included) and the dense mass matrix at qpos0 summed by the compiler
    on the unfused MJCF tree (the `M0` the fused runtime model must reproduce)."""
import hashlib
import json
import os
import sys
import xml.etree.ElementTree as ET

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from gymnasium_robotics_b200.mjcf import compile_mjcf  # noqa: E402
from gymnasium_robotics_b200.models import MODEL_OVERRIDES, MODEL_SOURCES, REFERENCE_ASSETS  # noqa: E402


def subtree_masses(path):
    out = {}

    def walk(b):
        tot = sum(float(i.get("mass")) for i in b.findall("inertial"))
        for ch in b.findall("body"):
            tot += walk(ch)
        out[b.get("name")] = tot
        return tot

    for b in ET.parse(path).getroot().iter("body"):
        if b.get("name") not in out:
            walk(b)
    return out


robot_xml = os.path.join(REFERENCE_ASSETS, "fetch", "robot.xml")
gripper = next(b for b in ET.parse(robot_xml).getroot().iter("body") if b.get("name") == "robot0:gripper_link")
m = compile_mjcf(os.path.join(REFERENCE_ASSETS, MODEL_SOURCES["fetch_pick_and_place"]))
out = {
    "blob_sha256": {name: hashlib.sha256(compile_mjcf(os.path.join(REFERENCE_ASSETS, rel), overrides=MODEL_OVERRIDES.get(name)).to_blob()).hexdigest()
                    for name, rel in MODEL_SOURCES.items()},
    "fetch_robot_xml": {"subtree_mass": subtree_masses(robot_xml),
                        "gripper_link_inertial_pos": [float(x) for x in gripper.find("inertial").get("pos").split()]},
    "fetch_pick_and_place_mjcf": {"bodies": len(m._full.bodies), "M0": m._full_arrays["M0"].tolist()},
}
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "fetch_model_facts.json"), "w") as f:
    json.dump(out, f, indent=0, sort_keys=True)
print(len(out["blob_sha256"]), "blobs")
