#!/usr/bin/env python
"""Generates tests/golden/ref_recipe_*.npz and the extra ref_optimization_* cases by EXECUTING THE
REFERENCE'S OWN STATEMENTS, lifted by AST from the files of the upstream project.

Needs a checkout of the upstream project (commit 74ae92b8) named by GACCUM_REFERENCE_DIR.  TensorFlow is
not a dependency of this project, so the lifted statements run against oracle/tf_stub (numpy fp32 emulation;
tests/golden/MANIFEST.json lists which stub primitives are restatements of TensorFlow rather than of the
reference).

What is lifted, verbatim (ast nodes selected by line number, compiled, exec'd -- never retyped):
  * distributedExample/02_single_worker_with_estimator_gaccum.py  model_fn lines 38-41 (hyper-parameters,
    `optimizer = tf.compat.v1.train.AdamOptimizer(...)`) and 47-73 (the whole accumulation recipe up to
    `train_op = tf.group(train_op, [tf.assign_add(global_step, 1)])`)
  * distributedExample/04_multi_worker_with_estimator_gaccum.py   model_fn lines 38-42 and 48-74
    (accumulators with aggregation=SUM; one replica here, so the all-reduce is the identity)
  * another-example.py  the nested function `_train_op_fn` (lines 126-155), called with a loss
Only the model / loss / metric lines between them are left out (the loss is a symbolic stand-in: under the
stub `tf.gradients` returns fed placeholders, the model's backward pass is not on this path).

Two further variant-A cases run optimization.py with ONE documented edit: the literal at line 76
(`gradient_accumulation_multiplier = 8`, a local of create_optimizer) is replaced through the AST by N=4 /
N=3; nothing else changes.  A third calls the reference's AdamWeightDecayOptimizer.apply_gradients directly
with a (None, var) pair, the only way the reference's `if grad is None` branch (optimization.py:132-133) can
execute (through create_optimizer a None gradient raises in assign_add, in TF and in the stub alike).

    GACCUM_REFERENCE_DIR=<checkout> python tests/golden/make_golden_recipes.py          # rewrites the fixtures + MANIFEST entries
"""
import ast
import importlib
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REFERENCE = os.environ.get("GACCUM_REFERENCE_DIR", "")     # checkout of the upstream project
SEED0 = 19830610

MNIST = [("conv2d/kernel", (3, 3, 1, 32)), ("conv2d/bias", (32,)), ("dense/kernel", (5408, 64)), ("dense/bias", (64,)),
         ("dense_1/kernel", (64, 10)), ("dense_1/bias", (10,))]                       # 02:22-28
SMALL = [("dense/kernel", (13, 7)), ("dense/bias", (7,)), ("dense_1/kernel", (7, 3)), ("dense_1/bias", (3,)), ("scalar_like", (1,))]
MINI_BERT = [
    ("bert/embeddings/word_embeddings", (37, 8)),
    ("bert/embeddings/LayerNorm/beta", (8,)),
    ("bert/embeddings/LayerNorm/gamma", (8,)),
    ("bert/encoder/layer_0/attention/self/query/kernel", (8, 8)),
    ("bert/encoder/layer_0/attention/self/query/bias", (8,)),
    ("bert/encoder/layer_0/output/layer_norm_like/scale", (5,)),
    ("output_weights", (2, 8)),
    ("output_bias", (2,)),
]
SUBSAMPLE_ABOVE, STRIDE = 4096, 61       # tensors larger than this are stored as every 61st element + their fp64 sum


def _tf():
    stub = os.path.join(ROOT, "oracle", "tf_stub")
    if stub not in sys.path:
        sys.path.insert(0, stub)
    sys.modules.pop("tensorflow", None)
    tf = importlib.import_module("tensorflow")
    assert "stub" in tf.__version__
    tf.reset_default_graph()
    return tf


def _init_vars(tf, variables, rng):
    init = {}
    for vname, shape in variables:
        if vname.endswith(("gamma", "scale")):
            val = np.ones(shape, np.float32)
        elif vname.endswith(("beta", "bias")):
            val = np.zeros(shape, np.float32)
        else:
            val = (rng.standard_normal(shape, dtype=np.float32) * np.float32(0.05)).astype(np.float32)
        init[vname] = val
        tf.get_variable(vname, shape=list(shape), dtype=tf.float32, initializer=val)
    return init


def _lift(path, func_path, line_ranges):
    """ast statements of function `func_path` (e.g. ["model_fn"]) whose first line is in one of line_ranges"""
    with open(path) as f:
        src = f.read()
    tree = ast.parse(src, filename=path)
    body = tree.body
    node = None
    for name in func_path:
        node = next(n for n in body if isinstance(n, ast.FunctionDef) and n.name == name)
        body = node.body
    picked = [st for st in body if any(lo <= st.lineno <= hi for lo, hi in line_ranges)]
    mod = ast.Module(body=picked, type_ignores=[])
    lines = [(st.lineno, st.end_lineno) for st in picked]
    return compile(mod, path, "exec"), lines


def _store(out, key, arr):
    arr = np.asarray(arr)
    if arr.size > SUBSAMPLE_ABOVE:
        out[key + "@sub"] = arr.reshape(-1)[::STRIDE].copy()
        out[key + "@sum"] = np.float64(arr.astype(np.float64).sum())
    else:
        out[key] = arr.copy()


def grads_for(variables, sigma, seed, step):
    """the gradients a consumer of the fixture must regenerate: PCG64(SEED0 + 7919*seed + step), float32 ziggurat"""
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + step))
    return [rng.standard_normal(shape, dtype=np.float32) * np.float32(sigma) for _, shape in variables]


def run_recipe(case, ref_file, func_path, line_ranges, namespace_fn, variables, N, lr, sigma, seed, steps, call=None):
    tf = _tf()
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + 100000))
    init = _init_vars(tf, variables, rng)
    tf.train.get_or_create_global_step()                # the Estimator creates it before model_fn runs
    code, lifted = _lift(os.path.join(REFERENCE, ref_file), func_path, line_ranges)
    ns = {"tf": tf}
    ns.update(namespace_fn(tf))
    exec(code, ns)
    train_op = call(ns, tf) if call else ns["train_op"]
    by_name = {v.name: v for v in tf.global_variables()}
    grad_ph = {p.name[len("grad/"):]: p for p in tf._g.placeholders}
    accum_vars = [v for v in tf.global_variables() if v.name.startswith("Variable_")]
    assert len(accum_vars) == len(variables)
    out = {"names": np.array([n for n, _ in variables]), "shapes": np.array([json.dumps(list(s)) for _, s in variables]),
           "N": N, "steps": steps, "lr": lr, "sigma": sigma, "seed": seed}
    for vname, val in init.items():
        _store(out, f"init/{vname}", val)
    sess = tf.Session()
    record = set(range(steps)) if sum(int(np.prod(s)) for _, s in variables) <= 65536 else {steps - 1, steps - 2}
    for s in range(steps):
        gl = grads_for(variables, sigma, seed, s)
        sess.run(train_op, feed_dict={grad_ph[vname + ":0"]: g for (vname, _), g in zip(variables, gl)})
        if s in record:
            for i, (vname, _) in enumerate(variables):
                _store(out, f"param/{s}/{vname}", by_name[vname + ":0"].value)
                _store(out, f"accum/{s}/{vname}", accum_vars[i].value)
                _store(out, f"m/{s}/{vname}", by_name[vname + "/Adam:0"].value)
                _store(out, f"v/{s}/{vname}", by_name[vname + "/Adam_1:0"].value)
            out[f"beta1_power/{s}"] = np.float32(by_name["Adam/beta1_power:0"].value)
            out[f"beta2_power/{s}"] = np.float32(by_name["Adam/beta2_power:0"].value)
        out[f"global_step/{s}"] = np.int64(by_name["global_step:0"].value)
    out["recorded_steps"] = np.array(sorted(record))
    path = os.path.join(HERE, f"ref_recipe_{case}.npz")
    np.savez_compressed(path, **out)
    return path, lifted


def _optimization_module(tf, N_override=None):
    """the reference's optimization.py as a module; optionally with the literal at line 76 replaced"""
    path = os.path.join(REFERENCE, "optimization.py")
    with open(path) as f:
        tree = ast.parse(f.read(), filename=path)
    edits = []
    if N_override is not None:
        for node in ast.walk(tree):
            if (isinstance(node, ast.Assign) and node.lineno == 76 and isinstance(node.targets[0], ast.Name)
                    and node.targets[0].id == "gradient_accumulation_multiplier" and isinstance(node.value, ast.Constant)):
                edits.append((node.lineno, node.value.value, N_override))
                node.value = ast.copy_location(ast.Constant(N_override), node.value)
        assert len(edits) == 1, "optimization.py:76 is not `gradient_accumulation_multiplier = <literal>`"
    mod = types.ModuleType("optimization_ref")
    mod.__file__ = path
    sys.modules["tensorflow"] = tf
    exec(compile(tree, path, "exec"), mod.__dict__)
    return mod, edits


def run_optimization_case(case, N, init_lr, num_train_steps, num_warmup_steps, sigma, seed, steps):
    tf = _tf()
    ref, edits = _optimization_module(tf, N_override=N)
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + 100000))
    init = _init_vars(tf, MINI_BERT, rng)
    train_op = ref.create_optimizer(tf.constant(0.0), init_lr, num_train_steps, num_warmup_steps, False)
    by_name = {v.name: v for v in tf.global_variables()}
    grad_ph = {p.name[len("grad/"):]: p for p in tf._g.placeholders}
    accum_vars = [v for v in tf.global_variables() if v.name.startswith("Variable_")]
    out = {"names": np.array([n for n, _ in MINI_BERT]), "N": N, "steps": steps, "init_lr": init_lr,
           "num_train_steps": num_train_steps, "num_warmup_steps": num_warmup_steps}
    for vname, val in init.items():
        out[f"init/{vname}"] = val
    sess = tf.Session()
    for s in range(steps):
        gl = grads_for(MINI_BERT, sigma, seed, s)
        feeds = {}
        for (vname, _), g in zip(MINI_BERT, gl):
            out[f"grad/{s}/{vname}"] = g
            feeds[grad_ph[vname + ":0"]] = g
        sess.run(train_op, feed_dict=feeds)
        for i, (vname, _) in enumerate(MINI_BERT):
            out[f"param/{s}/{vname}"] = by_name[vname + ":0"].value.copy()
            out[f"accum/{s}/{vname}"] = accum_vars[i].value.copy()
            out[f"m/{s}/{vname}"] = by_name[vname + "/adam_m:0"].value.copy()
            out[f"v/{s}/{vname}"] = by_name[vname + "/adam_v:0"].value.copy()
        out[f"global_step/{s}"] = np.int64(by_name["global_step:0"].value)
    path = os.path.join(HERE, f"ref_optimization_{case}.npz")
    np.savez_compressed(path, **out)
    return path, edits


def bert_small_manifest():
    """BASELINE config 2 shapes (upstream BERT L4_H512_A8 variable names in creation order; SURVEY.md 8 size table: T=73, P=28 764 674)."""
    H, L, inter = 512, 4, 2048
    out = [("bert/embeddings/word_embeddings", (30522, H)), ("bert/embeddings/token_type_embeddings", (2, H)),
           ("bert/embeddings/position_embeddings", (512, H)), ("bert/embeddings/LayerNorm/beta", (H,)), ("bert/embeddings/LayerNorm/gamma", (H,))]
    for l in range(L):
        b = f"bert/encoder/layer_{l}/"
        for nm in ("query", "key", "value"):
            out += [(b + f"attention/self/{nm}/kernel", (H, H)), (b + f"attention/self/{nm}/bias", (H,))]
        out += [(b + "attention/output/dense/kernel", (H, H)), (b + "attention/output/dense/bias", (H,)),
                (b + "attention/output/LayerNorm/beta", (H,)), (b + "attention/output/LayerNorm/gamma", (H,)),
                (b + "intermediate/dense/kernel", (H, inter)), (b + "intermediate/dense/bias", (inter,)),
                (b + "output/dense/kernel", (inter, H)), (b + "output/dense/bias", (H,)),
                (b + "output/LayerNorm/beta", (H,)), (b + "output/LayerNorm/gamma", (H,))]
    out += [("bert/pooler/dense/kernel", (H, H)), ("bert/pooler/dense/bias", (H,)), ("output_weights", (2, H)), ("output_bias", (2,))]
    return out


BIG_STRIDE = 4099      # full-size fixture: every 4099th element + fp64 sum of every tensor above SUBSAMPLE_ABOVE


def run_optimization_case_full_size(case, N, init_lr, num_train_steps, num_warmup_steps, sigma, seed, steps):
    """optimization.py (literal at :76 replaced by N) on the BERT-Small shapes of BASELINE config 2.  Gradients and initial
    values are regenerated from seeds by the consumer; the state after the last two micro-steps is stored subsampled."""
    tf = _tf()
    ref, edits = _optimization_module(tf, N_override=N)
    variables = bert_small_manifest()
    assert len(variables) == 73 and sum(int(np.prod(s)) for _, s in variables) == 28764674
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + 100000))
    _init_vars(tf, variables, rng)
    train_op = ref.create_optimizer(tf.constant(0.0), init_lr, num_train_steps, num_warmup_steps, False)
    by_name = {v.name: v for v in tf.global_variables()}
    grad_ph = {p.name[len("grad/"):]: p for p in tf._g.placeholders}
    accum_vars = [v for v in tf.global_variables() if v.name.startswith("Variable_")]
    out = {"names": np.array([n for n, _ in variables]), "shapes": np.array([json.dumps(list(s)) for _, s in variables]),
           "N": N, "steps": steps, "init_lr": init_lr, "num_train_steps": num_train_steps, "num_warmup_steps": num_warmup_steps,
           "sigma": sigma, "seed": seed, "stride": BIG_STRIDE}

    def store(key, arr):
        arr = np.asarray(arr)
        if arr.size > SUBSAMPLE_ABOVE:
            out[key + "@sub"] = arr.reshape(-1)[::BIG_STRIDE].copy()
            out[key + "@sum"] = np.float64(arr.astype(np.float64).sum())
        else:
            out[key] = arr.copy()
    sess = tf.Session()
    prev = None
    for s in range(steps):
        gl = grads_for(variables, sigma, seed, s)
        sess.run(train_op, feed_dict={grad_ph[vname + ":0"]: g for (vname, _), g in zip(variables, gl)})
        if s >= steps - 2:
            cur = {(kind, vname): by_name[vname + sfx].value.copy() for vname, _ in variables
                   for kind, sfx in (("param", ":0"), ("m", "/adam_m:0"), ("v", "/adam_v:0"))}
            # an accumulate-only micro-step leaves param / m / v as they were: stored once, under the step before
            same = prev is not None and all(np.array_equal(cur[k], prev[k]) for k in cur)
            if same:
                out[f"same_as/{s}"] = np.int64(s - 1)
            for i, (vname, _) in enumerate(variables):
                if not same:
                    store(f"param/{s}/{vname}", cur["param", vname])
                store(f"accum/{s}/{vname}", accum_vars[i].value)
                if not same:
                    store(f"m/{s}/{vname}", cur["m", vname])
                    store(f"v/{s}/{vname}", cur["v", vname])
            prev = cur
        out[f"global_step/{s}"] = np.int64(by_name["global_step:0"].value)
    out["recorded_steps"] = np.array([steps - 2, steps - 1])
    path = os.path.join(HERE, f"ref_fullsize_{case}.npz")
    np.savez_compressed(path, **out)
    return path, edits


def run_direct_apply_with_none(case, lr, sigma, seed, steps):
    """AdamWeightDecayOptimizer.apply_gradients called directly with a (None, var) pair (optimization.py:132-133)"""
    tf = _tf()
    ref, _ = _optimization_module(tf)
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + 100000))
    init = _init_vars(tf, MINI_BERT, rng)
    tvars = tf.trainable_variables()
    opt = ref.AdamWeightDecayOptimizer(learning_rate=lr, weight_decay_rate=0.01, beta_1=0.9, beta_2=0.999, epsilon=1e-6,
                                       exclude_from_weight_decay=["LayerNorm", "layer_norm", "bias"])
    none_at = 3
    phs = [None if i == none_at else tf.placeholder(tf.float32, v.shape, name="grad/" + v.name) for i, v in enumerate(tvars)]
    train_op = opt.apply_gradients(zip(phs, tvars))
    by_name = {v.name: v for v in tf.global_variables()}
    out = {"names": np.array([n for n, _ in MINI_BERT]), "steps": steps, "lr": lr, "none_at": none_at}
    for vname, val in init.items():
        out[f"init/{vname}"] = val
    sess = tf.Session()
    for s in range(steps):
        gl = grads_for(MINI_BERT, sigma, seed, s)
        feeds = {}
        for i, ((vname, _), g) in enumerate(zip(MINI_BERT, gl)):
            if i != none_at:
                out[f"grad/{s}/{vname}"] = g
                feeds[phs[i]] = g
        sess.run(train_op, feed_dict=feeds)
        for i, (vname, _) in enumerate(MINI_BERT):
            out[f"param/{s}/{vname}"] = by_name[vname + ":0"].value.copy()
            if i != none_at:
                out[f"m/{s}/{vname}"] = by_name[vname + "/adam_m:0"].value.copy()
                out[f"v/{s}/{vname}"] = by_name[vname + "/adam_v:0"].value.copy()
    assert MINI_BERT[none_at][0] + "/adam_m:0" not in by_name      # the skipped pair creates no slots (:132-133 `continue`)
    path = os.path.join(HERE, f"ref_{case}.npz")
    np.savez_compressed(path, **out)
    return path


if __name__ == "__main__":
    if not os.path.isdir(REFERENCE):
        raise SystemExit("make_golden_recipes.py needs GACCUM_REFERENCE_DIR: a checkout of the upstream project")
    sys.path.insert(0, os.path.dirname(HERE))
    from golden_util import array_digests
    meta = {}
    ex02 = "distributedExample/02_single_worker_with_estimator_gaccum.py"
    ex04 = "distributedExample/04_multi_worker_with_estimator_gaccum.py"

    def ns02(N, lr):
        return lambda tf: {"params": {"learning_rate": lr, "batch_size": 100, "gradient_accumulation_multiplier": N},
                           "loss": tf.constant(0.0)}

    def ns04(N, lr):
        return lambda tf: {"params": {"learning_rate": lr, "batch_size": 100, "gradient_accumulation_multiplier": N, "num_workers": 1},
                           "loss": tf.constant(0.0)}

    recipes = [
        # case, file, function path, line ranges, namespace, variables, N, lr, sigma, seed, steps, call
        ("02_small_n2", ex02, ["model_fn"], [(38, 41), (47, 73)], ns02(2, 1e-4), SMALL, 2, 1e-4, 0.5, 21, 9, None),         # 02:110 hparams: lr 1e-4, N=2
        ("02_mnist_n4", ex02, ["model_fn"], [(38, 41), (47, 73)], ns02(4, 1e-4), MNIST, 4, 1e-4, 0.1, 22, 10, None),        # BASELINE config 1 shapes, accum x4
        ("04_small_n2", ex04, ["model_fn"], [(38, 42), (48, 74)], ns04(2, 1e-4), SMALL, 2, 1e-4, 0.5, 23, 9, None),
        ("another_example_n3", "another-example.py", ["model_fn"], [(126, 155)],
         lambda tf: {"gradient_accumulation_multiplier": 3}, SMALL, 3, 1e-3, 0.5, 24, 11,                                   # a-e:135 default lr 1e-3, a-e:276 N=3
         lambda ns, tf: ns["_train_op_fn"](tf.constant(0.0))),
    ]
    for case, f, fp, lr_, nsf, variables, N, lr, sigma, seed, steps, call in recipes:
        path, lifted = run_recipe(case, f, fp, lr_, nsf, variables, N, lr, sigma, seed, steps, call)
        meta["recipe_" + case] = {"file": os.path.basename(path), "reference_file": f, "lifted_statement_lines": lifted,
                                  "N": N, "lr": lr, "sigma": sigma, "seed": seed, "steps": steps}
        print("wrote", path, "lifted", lifted)
    for case, N, cfg in (("n4_clipped", 4, (5e-3, 1000, 0, 0.5, 31, 10)), ("n3_warmup", 3, (1e-2, 40, 5, 0.2, 32, 8))):
        path, edits = run_optimization_case(case, N, *cfg)
        meta[case] = {"file": os.path.basename(path), "reference_file": "optimization.py",
                      "edits": [f"line {ln}: literal {old} -> {new} (AST)" for ln, old, new in edits], "config": cfg}
        print("wrote", path, edits)
    # BASELINE config 2 at full size: accum x4, README schedule shortened so that the run crosses the warm-up end; sigma 1e-3 => clipped
    path, edits = run_optimization_case_full_size("bert_small_n4", 4, 2e-5, 207900, 6, 1e-3, 41, 10)
    meta["fullsize_bert_small_n4"] = {"file": os.path.basename(path), "reference_file": "optimization.py",
                                      "edits": [f"line {ln}: literal {old} -> {new} (AST)" for ln, old, new in edits],
                                      "shapes": "BERT-Small L4_H512 (T=73, P=28 764 674)", "stored": f"last two micro-steps, every {BIG_STRIDE}th element + fp64 sums; param / m / v of the "
                                                "accumulate-only last step once, under the step before (same_as/<step>)",
                                      "config": [2e-5, 207900, 6, 1e-3, 41, 10]}
    print("wrote", path)
    path = run_direct_apply_with_none("direct_apply_none_grad", 1e-3, 0.3, 33, 3)
    meta["direct_apply_none_grad"] = {"file": os.path.basename(path), "reference_file": "optimization.py (unmodified)",
                                      "what": "AdamWeightDecayOptimizer.apply_gradients(zip(grads, tvars)) with grads[3] = None (:132-133)"}
    print("wrote", path)
    for entry in meta.values():
        entry["digests"] = array_digests(os.path.join(HERE, entry["file"]))
    man_path = os.path.join(HERE, "MANIFEST.json")
    with open(man_path) as fh:
        man = json.load(fh)
    man["recipe_generator"] = "tests/golden/make_golden_recipes.py"
    man["recipe_cases"] = meta
    man["stub_primitives_restating_tensorflow"] = {
        "tf.train.polynomial_decay": "TF 1.15 learning_rate_schedule.PolynomialDecay.__call__ (cycle=False)",
        "tf.clip_by_global_norm / tf.linalg.global_norm / tf.nn.l2_loss": "TF 1.15 clip_ops.py; l2_loss's reduction order is "
            "unspecified in TF -- stub AND oracle define it as the fp64-accumulated, once-rounded sum, so fixture and oracle agree "
            "by construction on that one point (tests hold 1e-5 against the CUDA path, whose order differs)",
        "tf.train.AdamOptimizer / tf.compat.v1.train.AdamOptimizer": "TF 1.15 adam.py + training_ops.cc ApplyAdam (dense, fp32, no nesterov)",
        "tf.cond / tf.group / tf.control_dependencies / Variable.assign(_add)": "graph-execution semantics (lazy dataflow, ref-variable reads)",
        "everything else": "one numpy fp32 ufunc per TF op; Python scalar -> tensor-dtype conversion as ops.convert_to_tensor",
    }
    man["what_is_the_reference's"] = ("op order, window logic, constants, conversion points, control dependencies, decay mask: executed from "
                                      "the reference's own statements (imported module or AST-lifted line ranges)")
    with open(man_path, "w") as fh:
        json.dump(man, fh, indent=1)
