"""Loader for tests/golden/ref_optimization_*.npz (made by tests/golden/make_golden.py)."""
import glob
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def array_digests(path):
    """sha256 per key family (the key up to its first '/') over every array's key, dtype, shape and bytes: the
    generators record these in MANIFEST.json from the upstream project's run, and tests hold the fixtures to them"""
    import hashlib
    z = np.load(path)
    h = {}
    for k in sorted(z.files):
        a = np.ascontiguousarray(z[k])
        h.setdefault(k.split("/")[0], hashlib.sha256()).update(f"{k}|{a.dtype.str}|{a.shape}|".encode() + a.tobytes())
    return {fam: d.hexdigest() for fam, d in sorted(h.items())}


def cases():
    return sorted(os.path.basename(p)[len("ref_optimization_"):-4]
                  for p in glob.glob(os.path.join(GOLDEN_DIR, "ref_optimization_*.npz")))


class Golden:
    def __init__(self, name):
        self.z = np.load(os.path.join(GOLDEN_DIR, f"ref_optimization_{name}.npz"))
        self.names = [str(n) for n in self.z["names"]]
        self.N = int(self.z["N"])
        self.steps = int(self.z["steps"])
        self.init_lr = float(self.z["init_lr"])
        self.num_train_steps = int(self.z["num_train_steps"])
        self.num_warmup_steps = int(self.z["num_warmup_steps"])

    def init(self):
        return [self.z[f"init/{n}"].copy() for n in self.names]

    def grads(self, s):
        return [self.z[f"grad/{s}/{n}"] for n in self.names]

    def state(self, s, kind):
        """kind in param|accum|m|v; m/v are None before the first apply created them (step 0 applies)."""
        return [self.z[f"{kind}/{s}/{n}"] for n in self.names]

    def global_step(self, s):
        return int(self.z[f"global_step/{s}"])


# ---- fixtures made by tests/golden/make_golden_recipes.py (AST-lifted recipe statements of 02 / 04 / another-example) ----
SEED0 = 19830610
STRIDE = 61


def recipe_cases():
    return sorted(os.path.basename(p)[len("ref_recipe_"):-4] for p in glob.glob(os.path.join(GOLDEN_DIR, "ref_recipe_*.npz")))


def recipe_grads(variables, sigma, seed, step):
    """must match make_golden_recipes.grads_for: PCG64(SEED0 + 7919*seed + step), float32 ziggurat normals"""
    rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * seed + step))
    return [rng.standard_normal(shape, dtype=np.float32) * np.float32(sigma) for _, shape in variables]


class RecipeGolden:
    """Variant-B trajectory: tf.train.AdamOptimizer inside the reference's inline accumulation recipe."""

    def __init__(self, name):
        import json
        self.z = np.load(os.path.join(GOLDEN_DIR, f"ref_recipe_{name}.npz"))
        self.names = [str(n) for n in self.z["names"]]
        self.shapes = [tuple(json.loads(str(s))) for s in self.z["shapes"]]
        self.variables = list(zip(self.names, self.shapes))
        self.N, self.steps = int(self.z["N"]), int(self.z["steps"])
        self.lr, self.sigma, self.seed = float(self.z["lr"]), float(self.z["sigma"]), int(self.z["seed"])
        self.recorded = [int(s) for s in self.z["recorded_steps"]]

    def init(self):
        """initial values; large tensors are regenerated exactly as the generator made them"""
        rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * self.seed + 100000))
        out = []
        for n, shape in self.variables:
            if n.endswith(("gamma", "scale")):
                v = np.ones(shape, np.float32)
            elif n.endswith(("beta", "bias")):
                v = np.zeros(shape, np.float32)
            else:
                v = (rng.standard_normal(shape, dtype=np.float32) * np.float32(0.05)).astype(np.float32)
            self.check(f"init/{n}", v, exact=True)
            out.append(v)
        return out

    def grads(self, s):
        return recipe_grads(self.variables, self.sigma, self.seed, s)

    def check(self, key, got, exact=True, rtol=1e-5, atol=1e-8):
        """compare `got` with the fixture entry `key` (full tensor, or every 61st element + fp64 sum for large ones)"""
        got = np.asarray(got)
        if key in self.z.files:
            exp = self.z[key]
            ok = np.array_equal(got.reshape(exp.shape), exp) if exact else np.allclose(got.reshape(exp.shape), exp, rtol=rtol, atol=atol)
            assert ok, f"{key} differs from the reference run"
        else:
            sub, tot = self.z[key + "@sub"], float(self.z[key + "@sum"])
            mine = got.reshape(-1)[::getattr(self, "stride", STRIDE)]
            ok = np.array_equal(mine, sub) if exact else np.allclose(mine, sub, rtol=rtol, atol=atol)
            assert ok, f"{key} (subsample) differs from the reference run"
            s = float(got.astype(np.float64).sum())
            assert (s == tot) if exact else abs(s - tot) <= 1e-5 * max(abs(tot), 1e-12) + 1e-7, f"{key} (sum) differs"


class DirectApplyGolden:
    def __init__(self):
        self.z = np.load(os.path.join(GOLDEN_DIR, "ref_direct_apply_none_grad.npz"))
        self.names = [str(n) for n in self.z["names"]]
        self.steps, self.lr, self.none_at = int(self.z["steps"]), float(self.z["lr"]), int(self.z["none_at"])


class FullsizeGolden(RecipeGolden):
    """ref_fullsize_*.npz: the reference's optimization.py (N patched) on BASELINE-sized shapes; gradients and initial
    values are regenerated from seeds, the last two micro-steps are stored as every `stride`-th element + fp64 sums."""

    def __init__(self, name):
        import json
        self.z = np.load(os.path.join(GOLDEN_DIR, f"ref_fullsize_{name}.npz"))
        self.names = [str(n) for n in self.z["names"]]
        self.shapes = [tuple(json.loads(str(s))) for s in self.z["shapes"]]
        self.variables = list(zip(self.names, self.shapes))
        self.N, self.steps = int(self.z["N"]), int(self.z["steps"])
        self.init_lr, self.num_train_steps, self.num_warmup_steps = float(self.z["init_lr"]), int(self.z["num_train_steps"]), int(self.z["num_warmup_steps"])
        self.sigma, self.seed, self.stride = float(self.z["sigma"]), int(self.z["seed"]), int(self.z["stride"])
        self.recorded = [int(s) for s in self.z["recorded_steps"]]

    def check(self, key, got, **kw):
        """param / m / v of a recorded accumulate-only step are stored once, under the step before (`same_as/<step>`)"""
        kind, s, n = key.split("/", 2)
        if kind in ("param", "m", "v") and f"same_as/{s}" in self.z.files:
            key = f"{kind}/{int(self.z[f'same_as/{s}'])}/{n}"
        super().check(key, got, **kw)

    def init(self):
        rng = np.random.Generator(np.random.PCG64(SEED0 + 7919 * self.seed + 100000))
        out = []
        for n, shape in self.variables:
            if n.endswith(("gamma", "scale")):
                v = np.ones(shape, np.float32)
            elif n.endswith(("beta", "bias")):
                v = np.zeros(shape, np.float32)
            else:
                v = (rng.standard_normal(shape, dtype=np.float32) * np.float32(0.05)).astype(np.float32)
            out.append(v)
        return out
