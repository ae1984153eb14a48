#!/usr/bin/env python
"""What tests/test_integration.py compares the drop-in boundary against, taken from a checkout of the reference:

    python tests/golden/make_golden_integration.py <reference-checkout>       -> tests/golden/integration.json

  state_dicts         name -> (shape, dtype) of every state_dict entry of a model built by the reference's own blueprint
                      loader (libs/support/utils.py create_model_from_py) from the reference's blueprint file, for the
                      creation strings tests/test_integration.py uses
  shell_functions     the names of the functions defined after `. score/process.sh; . score/score.sh`
  extract_call_sites  every line of pytorch/pipeline/extract_xvectors_for_pytorch.sh that runs the hard-coded
                      extractor, with the option names passed to it there

Only names, shapes and option names are stored; no source text of the reference."""
import json
import os
import re
import subprocess
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from test_integration import BLUEPRINT_CASES, EXTRACTOR, POOLING_CASES, case_key, layout_of, snowdar_creation  # noqa: E402


def reference_layout(utils, ref, blueprint, creation):
    model = utils.create_model_from_py(os.path.join(ref, "pytorch/model", blueprint), creation)
    sys.modules.pop(blueprint[:-3], None)
    return layout_of(model)


def main(ref):
    for name, attrs in (("tkinter", {"N": "n"}), ("tkinter.messagebox", {"NO": "no"}), ("turtle", {"xcor": None})):
        m = types.ModuleType(name)           # libs/nnet/transformer imports these by accident (SURVEY 8c)
        m.__dict__.update(attrs)
        m.__path__ = []
        sys.modules.setdefault(name, m)
    sys.path.insert(0, os.path.join(ref, "pytorch"))
    import libs.support.utils as utils
    cases = BLUEPRINT_CASES + [("snowdar_xvector.py", snowdar_creation(pooling, pp)) for pooling, pp in POOLING_CASES]
    sd = {case_key(b, c): reference_layout(utils, ref, b, c) for b, c in cases}

    r = subprocess.run(["bash", "-c", 'set -e; . "$1/score/process.sh"; . "$1/score/score.sh"; declare -F', "-", ref],
                       capture_output=True, text=True, check=True)
    functions = sorted(line.split()[2] for line in r.stdout.splitlines())

    sites = []
    with open(os.path.join(ref, "pytorch/pipeline/extract_xvectors_for_pytorch.sh")) as f:
        lines = f.read().splitlines()
    for i, line in enumerate(lines):
        if EXTRACTOR in line:
            j, command = i, line.split(EXTRACTOR, 1)[1]
            while command.rstrip().endswith("\\"):           # the command's continuation lines
                j += 1
                command = command.rstrip()[:-1] + " " + lines[j]
            sites.append({"line": i + 1, "options": re.findall(r"(?<!\S)(--[a-z][a-z-]*)", command)})

    out = {"state_dicts": sd, "shell_functions": functions, "extract_call_sites": sites}
    with open(os.path.join(HERE, "integration.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("integration.json ok:", {k: len(v) for k, v in out.items()})


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(os.path.abspath(sys.argv[1]))
