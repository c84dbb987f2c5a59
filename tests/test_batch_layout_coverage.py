"""Every step-kernel instantiation compiled in csrc/ is run by tests/test_gpu_batch_layout.py (no GPU needed): a new (build, W, NVP)
cannot land without a case that launches it, or an entry in that module's UNREACHABLE table saying why none can."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "gymnasium_robotics_b200", "csrc")


def _pairs(body):
    return {(int(w), int(v)) for w, v in re.findall(r"X\(\s*(\d+)\s*,\s*(\d+)\s*\)", body)}


def _macro(src, name):
    """Bodies of every `#define name(X) ...` in src (line continuations joined), in order of appearance."""
    src = src.replace("\\\n", " ")
    return [m.group(1) for m in re.finditer(r"^#define\s+" + name + r"\(X\)(.*)$", src, re.M)]


def instantiated_variants():
    """{(build, W, NVP)} with the build codes of b200sim_kernel_variant (include/b200sim.h)."""
    read = lambda f: open(os.path.join(CSRC, f)).read()
    out = set()
    (arm,) = _macro(read("b200sim.cu"), "B200_FOR_ALL_VARIANTS")
    out |= {(0, w, v) for w, v in _pairs(arm)}
    (wide,) = _macro(read("b200sim_wide.cu"), "B200_WIDE_VARIANTS")
    out |= {(1, w, v) for w, v in _pairs(wide)}
    # b200sim_kitchen.cu: `#ifdef B200_KITCHEN_GROUPS` list (the groups and hull builds, which both define it) `#else` the flat list
    kitchen = read("b200sim_kitchen.cu")
    assert re.search(r"#ifdef B200_KITCHEN_GROUPS\s*\n#define B200_KITCHEN_VARIANTS", kitchen), "kitchen variant lists moved"
    groups, flat = _macro(kitchen, "B200_KITCHEN_VARIANTS")
    assert "B200_KITCHEN_GROUPS" in read("b200sim_kitchen_groups.cu") and "B200_KITCHEN_GROUPS" in read("b200sim_kitchen_hull.cu")
    out |= {(2, w, v) for w, v in _pairs(flat)}
    out |= {(b, w, v) for b in (3, 4) for w, v in _pairs(groups)}
    return out


def test_every_instantiation_has_a_gpu_case():
    from tests.test_gpu_batch_layout import CASES, UNREACHABLE

    inst = instantiated_variants()
    assert {b for b, _, _ in inst} == {0, 1, 2, 3, 4}, sorted(inst)     # the parser found every build's list
    covered = {(c["build"], w, c["nvp"]) for c in CASES.values() for w in c["ws"]}
    missing = sorted(inst - covered - set(UNREACHABLE))
    assert not missing, f"step-kernel instantiations that no case of tests/test_gpu_batch_layout.py launches: {missing}"
    assert not (covered - inst), f"cases list variants that are not compiled: {sorted(covered - inst)}"
    for v, why in UNREACHABLE.items():
        assert v in inst and why.strip(), v
