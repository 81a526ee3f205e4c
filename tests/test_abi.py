"""The C-ABI library loads on a CPU-only box and exports every symbol include/lhw_b200.h declares
(no compute calls here)."""
import ctypes
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "lhw_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lhw_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import __graft_entry__
    __graft_entry__.build()
    from learninghumanoidwalking_b200 import _lib
    L = ctypes.CDLL(_lib.LIB_PATH)
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/lhw_b200.h but not exported"
    assert set(_lib.SIGNATURES) == set(names), set(_lib.SIGNATURES) ^ set(names)
    assert L.lhw_version() == 3   # 2: + Unitree H1 standing model; 3: + JVRC-1 stepping model, lhw_sim_set_step_height


def test_product_fails_loudly_without_cuda():
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from learninghumanoidwalking_b200 import _lib
    from learninghumanoidwalking_b200.envs import BatchedHumanoidEnv
    with pytest.raises(_lib.LhwError):
        BatchedHumanoidEnv(4)


def test_product_never_imports_the_oracle():
    """No product source may import, include, link or dlopen anything under oracle/ (comments may mention it)."""
    pkg = os.path.join(ROOT, "learninghumanoidwalking_b200")
    bad = re.compile(r"(^\s*(from|import)\s+oracle\b)|(#include\s*[\"<][^\">]*oracle)|liboracle|sim_oracle|ppo_oracle", re.M)
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                src = open(os.path.join(d, f)).read()
                assert not bad.search(src), f"{f} reaches into oracle/"


def test_run_experiment_keeps_the_reference_flags():
    """run_experiment.py (repo root) accepts every flag of the reference's entry point (run_experiment.py:152-260).  The flag
    list below was read off the reference; where LHW_REFERENCE names a checkout of it, it is re-derived from the file itself."""
    src = open(os.path.join(ROOT, "run_experiment.py")).read()
    ours = set(re.findall(r"\(\"(--[a-z-]+)\",", src))
    ref_flags = {"--env", "--logdir", "--input-norm-steps", "--n-itr", "--lr", "--eps", "--gamma", "--lam", "--std-dev",
                 "--learn-std", "--entropy-coeff", "--clip", "--minibatch-size", "--epochs", "--num-procs", "--max-grad-norm",
                 "--max-traj-len", "--no-mirror", "--mirror-coeff", "--eval-freq", "--continued", "--recurrent", "--imitate",
                 "--imitate-coeff", "--yaml", "--device", "--seed", "--path", "--out-dir", "--ep-len"}
    ref = os.environ.get("LHW_REFERENCE")
    if ref:
        assert set(re.findall(r"\"(--[a-z-]+)\"", open(os.path.join(ref, "run_experiment.py")).read())) == ref_flags
    assert ref_flags <= ours, ref_flags - ours


def test_torch_ops_library_registers_every_entry_point_and_rejects_bad_tensors():
    """csrc/torch_ops.cpp (TORCH_LIBRARY): torch.ops.lhw.* exist after loading liblhw_b200_torch.so, and their argument checks
    fire before anything reaches a kernel — here with CPU tensors (no GPU needed to see the TORCH_CHECK messages)."""
    import pytest
    import torch
    import __graft_entry__
    __graft_entry__.build()
    from learninghumanoidwalking_b200 import _lib
    O = _lib.ops()
    for name in ("sim_reset", "sim_step", "gae", "adv_stats", "adv_stats_from_gae", "adv_apply", "gather_minibatch", "grad_sumsq", "clip_adam_dev",
                 "fused_exchange", "ppo_loss", "linear_wgrad"):
        assert hasattr(O, name), name
    r = torch.zeros(4, 3)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        O.gae(r, r, r.int(), r, torch.zeros(3), r.clone(), 0.99, 0.95, None)
    with pytest.raises(RuntimeError, match="null sim handle"):
        O.sim_step(0, r, r.int(), 0, 0, r, 400, True, r, None, r, None, r.int(), r.int(), None, None)
    with pytest.raises(RuntimeError, match="null comm handle"):
        O.fused_exchange(0, r, r, r, 0, 3e-4, 0.9, 0.999, 1e-5, 0.5)
    with pytest.raises(RuntimeError, match="must be a CUDA tensor"):
        O.linear_wgrad(r, r, torch.zeros(3, 3), None, torch.zeros(64))
    with pytest.raises(RuntimeError, match="must share their rows"):
        O.linear_wgrad(r, torch.zeros(5, 3), torch.zeros(3, 3), None, torch.zeros(64))
    # the workspace query is host arithmetic: slices x (N*K + N) floats, a few hundred slices at most, nothing for an empty problem
    L = _lib.lib()
    for M, N, K in ((43690, 256, 256), (21845, 256, 37), (21845, 1, 256), (5, 3, 7)):
        w = L.lhw_linear_wgrad_workspace_floats(M, N, K)
        assert w % (N * K + N) == 0 and 1 <= w // (N * K + N) <= 300, (M, N, K, w)
    assert L.lhw_linear_wgrad_workspace_floats(0, 4, 4) == 0
