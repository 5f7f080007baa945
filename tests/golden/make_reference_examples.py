#!/usr/bin/env python
"""Generates reference_examples.json: what tests/test_model_compiler.py checks the config loader and the model compiler against.

    python tests/golden/make_reference_examples.py <checkout of the original mppi-isaac project>

* files    : every example task YAML of the original project (examples/*/*.yaml) and the conf/ YAMLs those tasks compose
             (their mppi / isaacgym defaults and their actors), verbatim.
* urdf     : three of its URDFs compiled straight from its assets/ by mppi_isaac_b200.model.urdf.compile_urdf (mass, inertia about
             the body origin, link and DOF names); the shipped models_compiled/ blocks must equal them.
* scenes   : per example task, (nb, nu, nlinks, num_bodies) of the scene built from its conf/ AND its assets/, or the
             NotImplementedError a task out of scope raises.
"""
import glob
import json
import os
import sys

import yaml

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

URDFS = ("point_robot.urdf", "heijn/heijn.urdf", "panda_isaac/robots/franka_panda_stick.urdf")


def main(ref):
    from mppi_isaac_b200.model.blob import build_scene
    from mppi_isaac_b200.model.urdf import compile_urdf
    from mppi_isaac_b200.utils.config_store import load_actor_cfgs, load_config

    tasks = sorted(os.path.relpath(t, ref) for t in glob.glob(os.path.join(ref, "examples", "*", "*.yaml")))
    need = set(tasks) | {"conf/actors/panda_stick.yaml", "conf/actors/goal.yaml"}
    for t in tasks:
        with open(os.path.join(ref, t)) as f:
            top = yaml.safe_load(f)
        for item in top.get("defaults", []):
            need |= {f"conf/{group}/{name}.yaml" for group, name in item.items()}
        need |= {f"conf/actors/{a}.yaml" for a in top["actors"]}
    files = {}
    for rel in sorted(need):
        with open(os.path.join(ref, rel)) as f:
            files[rel] = f.read()

    urdf = {}
    for rel in URDFS:
        m = compile_urdf(os.path.join(ref, "assets", "urdf", rel))
        urdf[rel] = dict(mass=m.mass.tolist(), inertia_o=m.inertia_o.tolist(), link_names=list(m.link_names), dof_names=list(m.dof_names))

    conf = [os.path.join(ref, "conf")]
    scenes = {}
    for t in tasks:
        cfg = load_config(os.path.join(ref, t), conf)
        try:
            sc = build_scene(load_actor_cfgs(cfg.actors, conf), assets_dirs=[os.path.join(ref, "assets")],
                             substep=cfg.isaacgym.dt / cfg.isaacgym.substeps)
            scenes[t.split("/")[1]] = [sc.model.nb, sc.nu, sc.model.nlinks, sc.num_bodies]
        except NotImplementedError:
            scenes[t.split("/")[1]] = "NotImplementedError"

    with open(os.path.join(HERE, "reference_examples.json"), "w") as fh:
        json.dump(dict(source="original mppi-isaac project: conf/ and examples/ YAMLs, URDFs compiled from its assets/",
                       files=files, urdf=urdf, scenes=scenes), fh, indent=0)


if __name__ == "__main__":
    main(sys.argv[1])
