"""Host-side logic of libgaccum.so (no GPU): schedule, predicate, decay mask, plan layout, errors,
and that the library exports every symbol include/gaccum.h declares."""
import ctypes
import os
import re

import numpy as np
import pytest

import gaccum_b200 as g
import oracle_c
import oracle_np as onp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_symbols_are_exported():
    hdr = open(os.path.join(ROOT, "include", "gaccum.h")).read()
    names = re.findall(r"GACCUM_API\s+[\w\s\*]+?\b(gaccum_\w+)\s*\(", hdr)
    assert len(names) >= 18, names
    lib = ctypes.CDLL(g.lib_path())
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in gaccum.h but not exported: {missing}"
    assert g.version() == 200


def test_library_has_no_torch_or_oracle_dependency():
    import subprocess
    out = subprocess.run(["ldd", g.lib_path()], capture_output=True, text=True).stdout
    assert "torch" not in out and "oracle" not in out and "python" not in out


def test_library_reads_no_gaccum_environment_variables():
    """Every kernel configuration is fixed at build time: the environment a process inherits cannot select an
    untested one.  A getenv("GACCUM_...") would leave its name as a NUL-terminated string in the binary."""
    with open(g.lib_path(), "rb") as f:
        blob = f.read()
    names = re.findall(rb"(?<=\x00)GACCUM_[A-Z0-9_]+(?=\x00)", blob)
    assert not names, f"libgaccum.so names environment variables: {sorted(set(names))}"


@pytest.mark.parametrize("sched", [(2e-5, 207900, 20790), (2e-5, 207900, 0), (1e-2, 12, 3), (5e-5, 1000, 100)])
def test_learning_rate_matches_both_oracles_bitwise(sched):
    init_lr, T, W = sched
    steps = list(range(0, 40)) + [W - 1, W, W + 1, T - 1, T, T + 5, 100000, 2**31 - 1 if T > 2**20 else T * 3]
    for s in steps:
        if s < 0:
            continue
        a = np.float32(g.learning_rate(init_lr, T, W, s))
        assert a == onp.learning_rate(init_lr, T, W, s), (sched, s)
        assert a == oracle_c.learning_rate(init_lr, T, W, s), (sched, s)


def test_apply_predicate_is_pre_increment_int32():
    assert [g.is_apply_step(s, 4) for s in range(9)] == [True, False, False, False, True, False, False, False, True]
    assert g.is_apply_step(0, 1) and g.is_apply_step(7, 1)
    assert g.is_apply_step(2**32, 8)              # cast to int32 first (optimization.py:77)
    assert not g.is_apply_step(5, 0)              # guarded: never divide by zero


def test_decay_mask_matches_reference_regex_logic():
    names = [n for n, _ in onp.MANIFESTS["bert_small"]()] + ["x/layer_norm/w:0", "dense/bias:12", "a:b", "plain"]
    got = g.decay_mask(names, 0.01)
    exp = [onp.do_use_weight_decay(onp.get_variable_name(n), 0.01) for n in names]
    assert got == exp
    man = onp.MANIFESTS["bert_small"]()
    assert sum(int(np.prod(sh)) for (_, sh), d in zip(man, got[:73]) if not d) == 28162   # SURVEY.md 8 size table
    assert g.decay_mask(names, 0.0) == [False] * len(names)               # `if not self.weight_decay_rate`
    assert g.decay_mask(["a/bias"], 0.01, exclude=[]) == [True]
    assert g.decay_mask(["layer_3/w", "layer_12/w"], 0.01, exclude=[r"layer_[0-9]+/"]) == [False, False]
    # the Python bindings evaluate the patterns with the reference's own engine (re.search, optimization.py:185):
    # Python-only syntax works exactly as it does in the reference
    assert g.decay_mask(["layer_3/w", "layer_x/w", "enc/w"], 0.01, exclude=[r"layer_\d+/", r"^(?!layer)"]) == [False, True, False]
    import re
    with pytest.raises(re.error):
        g.decay_mask(["a"], 0.01, exclude=["("])


def test_c_decay_mask_is_posix_ere_and_agrees_on_the_reference_patterns():
    """gaccum_decay_mask (for non-Python callers) speaks POSIX ERE: identical on the reference's plain substrings and
    on the common regex subset; Python-only syntax is documented as different (include/gaccum.h)."""
    from gaccum_b200 import _lib
    names = [n for n, _ in onp.MANIFESTS["bert_small"]()] + ["x/layer_norm/w:0", "dense/bias:12", "a:b", "plain"]
    assert _lib.decay_mask_c(names, 0.01) == g.decay_mask(names, 0.01)
    assert _lib.decay_mask_c(["layer_3/w", "layer_12/w"], 0.01, exclude=[r"layer_[0-9]+/"]) == [False, False]
    with pytest.raises(g.GaccumError):
        _lib.decay_mask_c(["a"], 0.01, exclude=["("])


@pytest.mark.parametrize("model,T,P", [("mnist_cnn", 6, 347146), ("bert_small", 73, 28764674),
                                       ("bert_base", 201, 109483778), ("bert_large", 393, 335143938)])
def test_plan_layout_for_baseline_configs(model, T, P):
    man = onp.MANIFESTS[model]()
    numels = [int(np.prod(s)) for _, s in man]
    plan = g.Plan(numels, [True] * T, g.HParams.bert(), device=-1)
    assert plan.T == T and plan.num_elements == P
    assert plan.algorithmic_bytes(False) == 12 * P and plan.algorithmic_bytes(True) == 36 * P
    off = plan.offsets
    assert off[0] == 0 and all(o % 32 == 0 for o in off)                       # 128-byte aligned slabs
    for i in range(T - 1):
        assert off[i + 1] == off[i] + (numels[i] + 31) // 32 * 32               # packed, no overlap
    assert plan.padded_size == off[-1] + (numels[-1] + 31) // 32 * 32
    assert plan.num_tiles == sum((n + 2047) // 2048 for n in numels)


def test_plan_edge_cases_and_errors():
    plan = g.Plan([0, 1, 0, 33], None, g.HParams.tf_adam(), device=-1)
    assert plan.offsets == [0, 0, 32, 32] and plan.padded_size == 96 and plan.num_tiles == 2
    empty = g.Plan([], None, g.HParams.bert(), device=-1)
    assert empty.padded_size == 0 and empty.num_tiles == 0
    with pytest.raises(g.GaccumError) as e:
        g.Plan([-1], None, g.HParams.bert(), device=-1)
    assert e.value.code == -1
    with pytest.raises(g.GaccumError):
        g.Plan([1] * 2000, None, g.HParams.bert(), device=-1)                 # > pointer-table capacity
    bad = g.HParams.bert(); bad.variant = 7
    with pytest.raises(g.GaccumError):
        g.Plan([4], None, bad, device=-1)


def test_no_cpu_fallback_compute_fails_loudly():
    """Without a device the product path must refuse, never compute."""
    plan = g.Plan([64], [True], g.HParams.bert(), device=-1)
    buf = np.zeros(64, np.float32)
    ptrs = g.Plan.ptr_array([buf.ctypes.data])
    args = g.StepArgs(0, 4, 0, 1e-3, 0.9, 0.999, 0.0)
    for call in (lambda: plan.step(ptrs, ptrs, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, args),
                 lambda: plan.accumulate(ptrs, buf.ctypes.data),
                 lambda: plan.apply(ptrs, ptrs, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, args),
                 lambda: plan.step_packed(buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, args)):
        with pytest.raises(g.GaccumError) as e:
            call()
        assert e.value.code == -2 and "no CPU fallback" in str(e.value)
    assert np.all(buf == 0)
    if g.device_count() == 0:
        with pytest.raises(g.GaccumError) as e:
            g.Plan([64], [True], g.HParams.bert(), device=0)
        assert e.value.code == -2


def test_train_op_rejects_cpu_tensors():
    import torch
    from gaccum_b200.train_op import GaccumTrainOp
    with pytest.raises(g.GaccumError):
        GaccumTrainOp([torch.zeros(4)], ["w"], g.HParams.bert(), 4, lambda s: 1e-3)


def test_create_optimizer_signature_and_tpu_rejection():
    import inspect
    from gaccum_b200 import optimization as opt
    assert list(inspect.signature(opt.create_optimizer).parameters) == \
        ["loss", "init_lr", "num_train_steps", "num_warmup_steps", "use_tpu"]           # optimization.py:25
    assert list(inspect.signature(opt.AdamWeightDecayOptimizer.__init__).parameters)[1:] == \
        ["learning_rate", "weight_decay_rate", "beta_1", "beta_2", "epsilon", "exclude_from_weight_decay", "name"]
    assert opt.gradient_accumulation_multiplier == 8                                     # optimization.py:76
    with pytest.raises(ValueError):
        opt.create_optimizer(lambda: None, 2e-5, 100, 10, True)
    o = opt.AdamWeightDecayOptimizer(1e-3, weight_decay_rate=0.01, exclude_from_weight_decay=["LayerNorm", "bias"])
    assert o._get_variable_name("a/b:0") == "a/b" and o._get_variable_name("a/b") == "a/b"
    assert o._do_use_weight_decay("x/kernel") and not o._do_use_weight_decay("x/bias") and not o._do_use_weight_decay("LayerNorm/g")


def test_product_manifests_match_the_oracles_and_the_survey():
    """bench.py takes shapes from the package, the tests from the oracle: they must be the same tables."""
    from gaccum_b200.manifests import MANIFESTS
    assert set(MANIFESTS) == set(onp.MANIFESTS)
    for k in MANIFESTS:
        assert MANIFESTS[k]() == onp.MANIFESTS[k]()
    assert len(MANIFESTS["bert_base"]()) == 201 and len(MANIFESTS["bert_large"]()) == 393


def test_oracle_is_not_imported_by_the_product():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may touch oracle/."""
    import subprocess, sys
    code = ("import sys, gaccum_b200, gaccum_b200.optimization, gaccum_b200.graph, gaccum_b200.manifests, "
            "gaccum_b200.estimator, gaccum_b200.distributed, gaccum_b200.train_op; "
            "bad=[m for m in sys.modules if m.startswith('oracle')]; print(bad); sys.exit(1 if bad else 0)")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    for rel in ("gradient-accumulation-tf-estimator_b200", "include", "examples"):
        for dp, _, files in os.walk(os.path.join(ROOT, rel)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cc")):
                    txt = open(os.path.join(dp, f), errors="ignore").read()
                    assert "import oracle" not in txt and "oracle_np" not in txt and "liboracle" not in txt, os.path.join(dp, f)


@pytest.mark.parametrize("model", ["mnist_cnn", "bert_small", "bert_large"])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_dp_shard_ranges_partition_the_tiles_evenly(model, world):
    """gaccum_dp_shard_range: contiguous, disjoint, covering tile ranges with near-equal element counts
    (the fused data-parallel apply gives each rank the tiles of one range)."""
    man = onp.MANIFESTS[model]()
    numels = [int(np.prod(s)) for _, s in man]
    plan = g.Plan(numels, None, g.HParams.bert(), device=-1)
    P, nt = plan.num_elements, plan.num_tiles
    prev_hi, total = 0, 0
    counts = []
    for r in range(world):
        lo, hi, n = plan.dp_shard_range(world, r)
        assert lo == prev_hi and hi >= lo
        prev_hi, total = hi, total + n
        counts.append(n)
    assert prev_hi == nt and total == P
    if nt >= 8 * world:
        assert max(counts) - min(counts) <= 2 * 2048 + max(numels) % 2048 + 2048     # within a couple of tiles
    with pytest.raises(g.GaccumError):
        plan.dp_shard_range(9, 0)
    with pytest.raises(g.GaccumError):
        plan.dp_shard_range(4, 4)
