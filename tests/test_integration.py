"""The drop-in boundary exercised from the REFERENCE's side (SURVEY 8b): the reference's blueprint loading (import the
blueprint file by path, evaluate the creation string) building the B200 blueprints and loading state_dicts laid out like
the reference's, and its shell function files with integration/score_b200.sh sourced on top.  What the reference defines
-- state_dict names, shapes and dtypes, shell function names, the extractor call sites of its job script -- is pinned in
tests/golden/integration.json (tests/golden/make_golden_integration.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXTRACTOR = "python3 subtools/pytorch/pipeline/onestep/extract_embeddings.py"

ECAPA_ARGS = ('80,10,training=False,extracted_embedding="near",'
              'ecapa_params={"channels":1024,"embd_dim":192,"mfa_conv":1536,'
              '"bn_params":{"momentum":0.5,"affine":True,"track_running_stats":True}},'
              'pooling="ecpa-attentive",pooling_params={"hidden_size":128,"time_attention":True,"stddev":True},'
              'fc1=False,fc2_params={"nonlinearity":"","nonlinearity_params":{"inplace":True},"bn-relu":False,'
              '"bn":True,"bn_params":{"momentum":0.5,"affine":False,"track_running_stats":True}}')
BLUEPRINT_CASES = [
    ("xvector.py", 'Xvector(23,10,training=False,extracted_embedding="far")'),
    ("ecapa_tdnn_xvector.py", "ECAPA_TDNN(" + ECAPA_ARGS + ")"),
]
POOLING_CASES = [
    ("multi-head", {"num_head": 4, "share": False}),
    ("multi-head", {"num_head": 2, "affine_layers": 2, "hidden_size": 32}),
    ("multi-resolution", {"num_head": 4, "temperature": True, "affine_layers": 1, "share": False}),
    ("multi-resolution", {"num_head": 3, "temperature": True, "affine_layers": 2, "share": False, "fixed": False}),
    ("attentive", {"affine_layers": 2, "context": [-1, 0, 1]}),
    ("lde", {"num_head": 5, "num_nodes": 64}),
    ("xi-postdist-softplus2", {"hidden_size": 32, "num_nodes": 64}),
]


def snowdar_creation(pooling, pp):
    return 'Xvector(40,10,training=False,pooling="{}",pooling_params={!r})'.format(pooling, pp)


def case_key(blueprint, creation):
    return blueprint + " " + creation


@pytest.fixture(scope="module")
def ref():
    with open(os.path.join(ROOT, "tests", "golden", "integration.json")) as f:
        return json.load(f)


def reference_state_dict(layout, seed):
    """Seeded values in the reference model's state_dict layout: name -> (shape, dtype)."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k, (shape, dtype) in sorted(layout.items()):
        dt = getattr(torch, dtype)
        sd[k] = (torch.randn(shape, generator=g).to(dt) if dt.is_floating_point
                 else torch.randint(0, 100, shape, generator=g).to(dt))
    return sd


def load_blueprint(blueprint, creation):
    """The reference's loader (utils.py:163-186), restated by the project's CLI: the B200 blueprint file is imported by
    path under its own module name and the creation string is evaluated in it."""
    from asv_subtools_b200.pipeline.extract_embeddings import create_model_from_py
    name, path = blueprint[:-3], os.path.join(ROOT, "asv_subtools_b200/model", blueprint)
    sys.modules.pop(name, None)                # same module name as the reference's blueprint: import ours
    try:
        return create_model_from_py(path, creation)
    finally:
        sys.path.remove(os.path.dirname(path))


def layout_of(model):
    return {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in model.state_dict().items()}


@pytest.mark.parametrize("blueprint,creation", BLUEPRINT_CASES)
def test_reference_loader_builds_b200_blueprints_and_loads_reference_state_dicts(ref, blueprint, creation):
    """The B200 blueprint file loads the way extract_embeddings.py:63 loads the reference's, with the reference's creation
    string, and a state_dict laid out like one made by the REFERENCE's own class (same names, shapes and dtypes) loads
    with strict=False: nothing missing, nothing unexpected; the plugin surface of framework.py is there."""
    layout = ref["state_dicts"][case_key(blueprint, creation)]
    sd = reference_state_dict(layout, 11)
    model = load_blueprint(blueprint, creation)
    assert type(model).__module__ == blueprint[:-3] and "asv_subtools_b200" in sys.modules[type(model).__module__].__file__
    assert layout_of(model) == layout
    res = model.load_state_dict(sd, strict=False)
    assert not res.missing_keys and not res.unexpected_keys
    k = next(k for k in sd if k.endswith("affine.weight"))
    assert torch.equal(model.state_dict()[k], sd[k])
    for attr in ("extract_embedding", "extracted_embedding", "eval", "train", "cuda", "cpu", "parameters"):
        assert hasattr(model, attr), attr
    assert next(model.parameters()).device.type == "cpu"       # utils.to_device reads this (utils.py:105-114)
    with pytest.raises(Exception):                             # no CPU path: extraction on a CPU-resident model raises
        model.eval().extract_embedding(np.zeros((50, 23 if "xvector.py" == blueprint else 80), dtype=np.float32))
    sys.modules.pop(blueprint[:-3], None)


def test_shell_shadows_cover_the_reference_functions_they_replace(ref):
    """After the reference's function files (scoreSets.sh:133-134, here one stub per function they define) and
    `. integration/score_b200.sh` (the one added line), every function the B200 file defines existed before under the
    same name, now runs the B200 CLI, and the functions it does not shadow (e.g. get_params, process) are still the
    reference's."""
    names = ref["shell_functions"]
    assert {"get_params", "process"} <= set(names)
    stubs = "".join("function {0}(){{ echo reference_{0}; }}\n".format(f) for f in names)
    script = r'''
set -e
{stubs}
before=$(declare -F | awk '{{print $3}}' | sort)
. {root}/integration/score_b200.sh
mine=$(grep -o '^function [a-z_]*' {root}/integration/score_b200.sh | awk '{{print $2}}' | grep -v '^_')
for f in $mine; do
  echo "$before" | grep -qx "$f" || {{ echo "NOT-IN-REFERENCE $f"; exit 3; }}
  declare -f $f | grep -q _xvb200 || {{ echo "NOT-SHADOWED $f"; exit 4; }}
done
for f in {names}; do
  echo "$mine" | grep -qx "$f" || declare -f $f | grep -q "reference_$f" || {{ echo "CHANGED $f"; exit 5; }}
done
echo OK $(grep -c '^function [a-z]' {root}/integration/score_b200.sh)
'''.format(stubs=stubs, root=ROOT, names=" ".join(names))
    r = subprocess.run(["bash", "-c", script], capture_output=True, text=True)
    assert r.returncode == 0 and r.stdout.startswith("OK"), r.stdout + r.stderr
    assert int(r.stdout.split()[1]) >= 12


def test_extraction_wrapper_rewrites_only_the_hard_coded_extractor_command(ref, tmp_path):
    """The wrapper on a job script whose extractor calls sit where the reference's extract_xvectors_for_pytorch.sh has
    them, with the same options: both calls (the --use-gpu and the CPU branch, :128 and :139) are rewritten to the batched
    CLI with their options kept."""
    sites = ref["extract_call_sites"]
    assert len(sites) == 2 and all("--use-gpu" in s["options"] for s in sites)
    lines = ["#!/bin/bash"] + ["# step %d" % i for i in range(2, max(s["line"] for s in sites) + 2)]
    for s in sites:
        lines[s["line"] - 1] = "  {} {} model feats output || exit 1".format(EXTRACTOR, " ".join(o + "=x" for o in s["options"]))
    job = tmp_path / "extract_xvectors_for_pytorch.sh"
    job.write_text("\n".join(lines) + "\n")
    env = dict(os.environ, XVB200_DRYRUN="1", XVB200_REF=str(job))
    r = subprocess.run(["bash", os.path.join(ROOT, "integration/extract_xvectors_b200.sh"), "m", "d", "o"], capture_output=True,
                       text=True, env=env, cwd=str(tmp_path))
    out = [l for l in r.stdout.splitlines() if l.startswith(">")]
    assert r.returncode == 0 and len(out) == len(sites), r.stdout + r.stderr
    for l, s in zip(out, sites):
        assert "-m asv_subtools_b200.pipeline.extract_embeddings --batch-size 256 --blueprint-dir" in l
        assert all(o + "=x" in l for o in s["options"]) and "onestep/extract_embeddings.py" not in l


@pytest.mark.parametrize("pooling,pp", POOLING_CASES)
def test_snowdar_pooling_variants_register_the_reference_parameters(ref, pooling, pp):
    """Every pooling option of the snowdar blueprint's switch (snowdar_xvector.py:119-136): the B200 blueprint registers the
    same parameter / buffer names and shapes as the reference's (grouped attention affines, temperatures, LDE dictionary,
    xi-vector prior), so reference checkpoints of those configurations load with strict=True."""
    creation = snowdar_creation(pooling, pp)
    layout = ref["state_dicts"][case_key("snowdar_xvector.py", creation)]
    ours = load_blueprint("snowdar_xvector.py", creation)
    assert layout_of(ours) == layout
    sd = reference_state_dict(layout, 12)
    assert not ours.load_state_dict(sd, strict=True).missing_keys
    assert all(torch.equal(ours.state_dict()[k], v) for k, v in sd.items())
    sys.modules.pop("snowdar_xvector", None)
