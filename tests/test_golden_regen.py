"""The committed golden fixtures are exactly what tests/golden/make_golden.py and make_golden_recipes.py produce
from the reference's own code.  The upstream project's source is not part of this repository, so the generators
record, from their run against it, a sha256 per key family of every fixture in MANIFEST.json: every committed
fixture is held to those digests.  With GACCUM_REFERENCE_DIR naming a checkout of the upstream project, the
generators also run again here and must reproduce the committed fixtures bit for bit."""
import glob
import importlib.util
import json
import os
import sys

import numpy as np

from golden_util import array_digests

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE_DIR = os.environ.get("GACCUM_REFERENCE_DIR", "")
HAVE_REFERENCE = bool(REFERENCE_DIR) and os.path.isfile(os.path.join(REFERENCE_DIR, "optimization.py"))
with open(os.path.join(HERE, "golden", "MANIFEST.json")) as _f:
    MANIFEST = json.load(_f)


def _holds_recorded_run(section):
    for name, e in MANIFEST[section].items():
        got = array_digests(os.path.join(HERE, "golden", e["file"]))
        assert got == e["digests"], f"{name}: {e['file']} differs from the upstream run in " + \
            str(sorted(k for k in set(got) | set(e["digests"]) if got.get(k) != e["digests"].get(k)))


def test_fixtures_regenerate_bit_identically(tmp_path, monkeypatch):
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(HERE, "golden", "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    assert set(MANIFEST["cases"]) == set(mg.CASES)
    _holds_recorded_run("cases")
    if not HAVE_REFERENCE:
        return
    monkeypatch.setattr(mg, "HERE", str(tmp_path))
    saved_path, saved_mods = list(sys.path), {k: sys.modules.get(k) for k in ("tensorflow", "optimization")}
    try:
        for name, cfg in mg.CASES.items():
            path, steps = mg.run_case(name, *cfg)
            new = np.load(path)
            old = np.load(os.path.join(HERE, "golden", os.path.basename(path)))
            assert set(new.files) == set(old.files)
            for k in new.files:
                assert np.array_equal(new[k], old[k]), f"{name}: {k} differs from the committed fixture"
    finally:
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_recipe_fixtures_regenerate_bit_identically(tmp_path, monkeypatch):
    """Same for tests/golden/make_golden_recipes.py: the AST-lifted statements of 02 / 04 / another-example and the
    N-patched optimization.py produce exactly the committed ref_recipe_* / ref_optimization_n* / ref_direct_* /
    ref_fullsize_* files; between them, the two generators' records cover every committed fixture."""
    recorded = {e["file"] for sec in ("cases", "recipe_cases") for e in MANIFEST[sec].values()}
    assert recorded == {os.path.basename(p) for p in glob.glob(os.path.join(HERE, "golden", "*.npz"))}
    _holds_recorded_run("recipe_cases")
    if not HAVE_REFERENCE:
        return
    spec = importlib.util.spec_from_file_location("make_golden_recipes", os.path.join(HERE, "golden", "make_golden_recipes.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    monkeypatch.setattr(mg, "HERE", str(tmp_path))
    saved_path, saved_mods = list(sys.path), {k: sys.modules.get(k) for k in ("tensorflow", "optimization")}
    try:
        made = []
        path, lifted = mg.run_recipe("02_small_n2", "distributedExample/02_single_worker_with_estimator_gaccum.py", ["model_fn"],
                                     [(38, 41), (47, 73)],
                                     lambda tf: {"params": {"learning_rate": 1e-4, "batch_size": 100, "gradient_accumulation_multiplier": 2},
                                                 "loss": tf.constant(0.0)}, mg.SMALL, 2, 1e-4, 0.5, 21, 9, None)
        assert lifted[0][0] == 38 and lifted[-1][1] == 73
        made.append(path)
        path, _ = mg.run_recipe("another_example_n3", "another-example.py", ["model_fn"], [(126, 155)],
                                lambda tf: {"gradient_accumulation_multiplier": 3}, mg.SMALL, 3, 1e-3, 0.5, 24, 11,
                                lambda ns, tf: ns["_train_op_fn"](tf.constant(0.0)))
        made.append(path)
        path, edits = mg.run_optimization_case("n3_warmup", 3, 1e-2, 40, 5, 0.2, 32, 8)
        assert edits == [(76, 8, 3)]
        made.append(path)
        made.append(mg.run_direct_apply_with_none("direct_apply_none_grad", 1e-3, 0.3, 33, 3))
        for path in made:
            new = np.load(path)
            old = np.load(os.path.join(HERE, "golden", os.path.basename(path)))
            assert set(new.files) == set(old.files), os.path.basename(path)
            for k in new.files:
                assert np.array_equal(new[k], old[k]), f"{os.path.basename(path)}: {k} differs from the committed fixture"
    finally:
        sys.path[:] = saved_path
        for k, v in saved_mods.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
