"""What the reference's two command-line callers write on its YCB example, kept as golden data.

The reference's own src/stocs_match_one_object.cpp and src/model_preprocess.cpp, built unmodified
against model_matching_b200/host, were checked to write the same files byte for byte and print the
same counters as this repository's model_preprocess / stocs_single run with the reference's quad
selection (STOCS_REF_SHUFFLE=1) and seed 7.  golden/ref_callers_ycb.json keeps those counters and
the size and SHA-256 of every file: the offline artefacts (model_search.ply, ppf_map), the pose file
and the debug clouds.  The CLIs run here as the reference's callers are run: the repository path they are given
does not exist and STOCS_PATH_REMAP redirects every file the shim opens under it."""
import hashlib
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "model_matching_b200", "host")
GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_callers_ycb.json")
COMPILED_IN = "/compiled/in/model_matching"    # stands for the path the reference's caller compiles in
STDOUT_NUMBERS = (r"\|M\| = (\d+)", r"\|map\(M\)\| = (\d+)", r"\|S\|: (\d+)", r"Sampled (\d+) bases",
                  r"found (\d+) congruent sets", r"Transforms to verify: (\d+)",
                  r"best index: (-?\d+), maximum score: ([0-9.e+-]+)")


@pytest.mark.gpu
def test_cli_reproduces_the_reference_callers_outputs(tmp_path):
    with open(GOLDEN) as f:
        g = json.load(f)
    obj, scene = g["object"], g["scene"]
    repo = str(tmp_path / "repo")
    scene_dir = os.path.join(repo, "examples", scene)
    shutil.copytree(os.path.join(ROOT, "tests", "golden", "examples", scene), scene_dir)
    os.makedirs(os.path.join(repo, "models", obj))
    shutil.copy(os.path.join(ROOT, "tests", "golden", "models", obj, "textured_vertices.ply"), os.path.join(repo, "models", obj))
    env = dict(os.environ, STOCS_REPO_PATH=COMPILED_IN, STOCS_PATH_REMAP=f"{COMPILED_IN}={repo}", **g["env"])
    p1 = subprocess.run([os.path.join(HOST, "model_preprocess"), obj], env=env, capture_output=True, text=True, timeout=300)
    assert p1.returncode == 0, p1.stdout + p1.stderr
    assert g["preprocess_line"] in p1.stdout
    p2 = subprocess.run([os.path.join(HOST, "stocs_single"), scene_dir, obj], env=env, capture_output=True, text=True, timeout=300)
    assert p2.returncode == 0, p2.stdout + p2.stderr
    assert [n for pat in STDOUT_NUMBERS for n in re.search(pat, p2.stdout).groups()] == g["stdout_numbers"]
    with open(os.path.join(scene_dir, f"best_pose_candidate_{obj}.txt")) as f:
        assert f.read().strip() == g["pose"]
    for rel, want in g["files"].items():
        with open(os.path.join(repo, rel), "rb") as f:
            data = f.read()
        assert {"sha256": hashlib.sha256(data).hexdigest(), "bytes": len(data)} == want, rel
