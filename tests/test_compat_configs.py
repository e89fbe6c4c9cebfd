"""CPU: the reference's own, unchanged ``configs/*.py`` drive the B200 modules through ``compat/`` (SURVEY 8b, north
star: "configs/*.py work unchanged").  Needs a checkout of the reference, which this repository does not contain: set
CPC_REFERENCE_ROOT to it (the test skips otherwise); the expected values come from the reference's own ``setup_model``
(tests/golden/configs_all.json, written by oracle/make_golden.py::golden_configs_all).  Follow-up: store the reference's
small configs/*.py files under tests/golden/ and point the worker at them, so that the test runs without a checkout."""
import json
import os
import subprocess
import sys

import pytest

from conftest import PKG, ROOT, load_golden

REFERENCE = os.environ.get("CPC_REFERENCE_ROOT", "")

WORKER = r'''
import json, sys
compat, pkg, oracle, reference = sys.argv[1:5]
sys.dont_write_bytecode = True
sys.path[:0] = [compat, pkg, reference]
import configs.experiment_configs as ec                      # the reference's file, resolved against compat/
import audio_model, scalogram_model, setup_functions
assert audio_model.__file__.startswith(compat) and scalogram_model.__file__.startswith(compat)
assert ec.__file__.startswith(reference)
import cpc_b200
assert ec.experiments['e24']['encoder_config']['model'] is cpc_b200.ScalogramResidualEncoder
assert ec.experiments['e24']['ar_model_config']['model'] is cpc_b200.ConvolutionalArModel
assert ec.experiments['e24']['training_config']['score_function'] is cpc_b200.linear_score_function
sys.path.append(oracle)
from make_golden import build_all_experiments
print("RESULT " + json.dumps(build_all_experiments(ec.experiments, setup_functions.setup_model)))
'''


@pytest.mark.skipif(not REFERENCE or not os.path.isfile(os.path.join(REFERENCE, "configs", "experiment_configs.py")),
                    reason="no reference checkout: set CPC_REFERENCE_ROOT to one")
def test_reference_configs_build_every_experiment_through_compat(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    out = subprocess.run([sys.executable, str(script), os.path.join(PKG, "compat"), PKG, os.path.join(ROOT, "oracle"),
                          REFERENCE], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    mine = json.loads([l for l in out.stdout.splitlines() if l.startswith("RESULT ")][0][len("RESULT "):])
    want = load_golden("configs_all.json")
    assert sorted(mine) == sorted(want)
    assert len(want) >= 35 and "e29" in want and "e32" in want
    for name, ref in want.items():
        got = mine[name]
        if "error" in ref:                                    # the reference itself cannot build this one
            continue
        assert "error" not in got, (name, got)
        assert got["item_length"] == ref["item_length"], name
        assert got["params"] == ref["params"], (name, set(got["params"]) ^ set(ref["params"]))
        assert got["buffers"] == ref["buffers"], name
        assert got["preprocessing"] == ref["preprocessing"], name
        assert (got["score_function"], got["encoder"], got["ar"]) == (ref["score_function"], ref["encoder"], ref["ar"]), name
