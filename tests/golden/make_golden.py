#!/usr/bin/env python
"""Generates tests/golden/ref_optimization_*.npz by EXECUTING THE REFERENCE'S OWN optimization.py.

Needs a checkout of the upstream project (hpandana/gradient-accumulation-tf-estimator, commit
74ae92b8) named by GACCUM_REFERENCE_DIR.  TensorFlow is not a dependency of this project, so the
reference file is imported unmodified with oracle/tf_stub first on sys.path (a numpy fp32 emulation
of the TF1 primitives it calls; see that package's docstring for exactly what this does and does
not pin).  For each case we build the
reference graph with `optimization.create_optimizer(loss, init_lr, num_train_steps,
num_warmup_steps, use_tpu=False)`, feed seeded gradients for 2*N+2 micro-steps (N = 8, hard-coded
at optimization.py:76) and record every variable after every `session.run(train_op)`.

    GACCUM_REFERENCE_DIR=<checkout> python tests/golden/make_golden.py          # rewrites the fixtures
"""
import importlib
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("GACCUM_REFERENCE_DIR", "")     # checkout of the upstream project

# mini-BERT: names drive the decay mask (LayerNorm / layer_norm / bias are excluded, :65)
VARIABLES = [
    ("bert/embeddings/word_embeddings", (37, 8)),
    ("bert/embeddings/LayerNorm/beta", (8,)),
    ("bert/embeddings/LayerNorm/gamma", (8,)),
    ("bert/encoder/layer_0/attention/self/query/kernel", (8, 8)),
    ("bert/encoder/layer_0/attention/self/query/bias", (8,)),
    ("bert/encoder/layer_0/output/layer_norm_like/scale", (5,)),
    ("output_weights", (2, 8)),
    ("output_bias", (2,)),
]

CASES = {
    # name: (init_lr, num_train_steps, num_warmup_steps, grad sigma, seed)
    "warmup_unclipped": (2e-5, 207900, 20790, 1e-3, 11),     # README.md:72,75 schedule; ||n|| << 1
    "nowarmup_clipped": (5e-3, 1000, 0, 0.5, 12),            # every apply clips
    "mixed_short_decay": (1e-2, 12, 3, 0.03, 13),            # crosses warm-up end and decay end (lr -> 0)
}


def run_case(name, init_lr, num_train_steps, num_warmup_steps, sigma, seed):
    sys.path.insert(0, os.path.join(ROOT, "oracle", "tf_stub"))
    sys.path.insert(1, REFERENCE)
    for m in ("tensorflow", "optimization"):
        sys.modules.pop(m, None)
    tf = importlib.import_module("tensorflow")
    assert "stub" in tf.__version__
    ref = importlib.import_module("optimization")
    assert os.path.realpath(ref.__file__) == os.path.join(REFERENCE, "optimization.py"), ref.__file__
    tf.reset_default_graph()
    rng = np.random.Generator(np.random.PCG64(19830610 + seed))
    init = {}
    tvars = []
    for vname, shape in VARIABLES:
        if vname.endswith("gamma") or vname.endswith("scale"):
            val = np.ones(shape, np.float32)
        elif vname.endswith("beta") or vname.endswith("bias"):
            val = np.zeros(shape, np.float32)
        else:
            val = rng.normal(0, 0.02, shape).astype(np.float32)
        init[vname] = val
        tvars.append(tf.get_variable(vname, shape=list(shape), dtype=tf.float32, initializer=val))
    loss = tf.constant(0.0)            # symbolic stand-in: tf.gradients() yields fed placeholders
    train_op = ref.create_optimizer(loss, init_lr, num_train_steps, num_warmup_steps, False)
    by_name = {v.name: v for v in tf.global_variables()}
    grad_ph = {p.name[len("grad/"):]: p for p in tf._g.placeholders}
    accum_vars = [v for v in tf.global_variables() if v.name.startswith("Variable_")]   # optimization.py:78 order
    assert len(accum_vars) == len(tvars)
    N = 8                                                     # optimization.py:76
    steps = 2 * N + 2
    out = {"names": np.array([n for n, _ in VARIABLES]), "N": N, "steps": steps,
           "init_lr": init_lr, "num_train_steps": num_train_steps, "num_warmup_steps": num_warmup_steps}
    for vname, val in init.items():
        out[f"init/{vname}"] = val
    sess = tf.Session()
    for s in range(steps):
        feeds = {}
        for i, (vname, shape) in enumerate(VARIABLES):
            g = rng.normal(0, sigma, shape).astype(np.float32)
            if s == 5 and i == 3:
                g[...] = 0.0                                   # an all-zero gradient tensor
            out[f"grad/{s}/{vname}"] = g
            feeds[grad_ph[vname + ":0"]] = g
        sess.run(train_op, feed_dict=feeds)
        for i, (vname, _) in enumerate(VARIABLES):
            out[f"param/{s}/{vname}"] = by_name[vname + ":0"].value.copy()
            out[f"accum/{s}/{vname}"] = accum_vars[i].value.copy()
            if vname + "/adam_m:0" in by_name:
                out[f"m/{s}/{vname}"] = by_name[vname + "/adam_m:0"].value.copy()
                out[f"v/{s}/{vname}"] = by_name[vname + "/adam_v:0"].value.copy()
        out[f"global_step/{s}"] = np.int64(by_name["global_step:0"].value)
    path = os.path.join(HERE, f"ref_optimization_{name}.npz")
    np.savez_compressed(path, **out)
    sys.path.remove(os.path.join(ROOT, "oracle", "tf_stub"))
    sys.path.remove(REFERENCE)
    return path, steps


if __name__ == "__main__":
    if not os.path.isdir(REFERENCE):
        raise SystemExit("make_golden.py needs GACCUM_REFERENCE_DIR: a checkout of the upstream project")
    sys.path.insert(0, os.path.dirname(HERE))
    from golden_util import array_digests
    meta = {}
    for name, cfg in CASES.items():
        path, steps = run_case(name, *cfg)
        meta[name] = {"file": os.path.basename(path), "steps": steps, "config": cfg, "digests": array_digests(path)}
        print("wrote", path)
    with open(os.path.join(HERE, "MANIFEST.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_golden.py", "reference_commit": "74ae92b8",
                   "reference_file": "optimization.py (imported unmodified)",
                   "tf": "oracle/tf_stub numpy emulation (TensorFlow not installable)", "cases": meta}, f, indent=1)
