"""CPU-side checks of the drop-in boundary: the C-ABI library builds/loads, exports every symbol
include/fi_learner.h declares, and fails loudly (no CPU fallback) when there is no CUDA device."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

import _util as U

HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")


def _declared_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"FI_API\s+[\w\s\*]+?\b(fi_\w+)\s*\(", src)))


def test_header_compiles_as_plain_c(tmp_path):
    c = tmp_path / "t.c"
    c.write_text('#include "fi_learner.h"\nint main(void){fi_learner_config c; fi_batch b; (void)c; (void)b; return 0;}\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.dirname(HEADER), str(c)], check=True)


def test_library_exports_every_declared_symbol(fi):
    lib = fi.load_library()
    declared = _declared_symbols()
    assert len(declared) >= 50
    missing = [s for s in declared if not hasattr(lib, s)]
    assert not missing, f"declared in fi_learner.h but not exported: {missing}"
    # and the ctypes table binds exactly the declared set
    from freeimpala_b200 import _lib
    assert sorted(_lib.SIGNATURES) == declared


def test_config_struct_layout_matches_header(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "s.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\nint main(void){printf("%zu %zu %zu %zu %zu\\n",'
                 'sizeof(fi_learner_config), offsetof(fi_learner_config, lr), offsetof(fi_learner_config, gemm_mode),'
                 'offsetof(fi_learner_config, checkpoint_location), sizeof(fi_batch));return 0;}\n')
    exe = tmp_path / "s"
    subprocess.run(["gcc", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    size, off_lr, off_gemm, off_ckpt, bsize = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert (C.sizeof(K), K.lr.offset, K.gemm_mode.offset, K.checkpoint_location.offset) == (size, off_lr, off_gemm, off_ckpt)
    assert C.sizeof(_lib.FiBatch) == bsize


def test_no_cpu_fallback_without_a_device(fi):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    with pytest.raises(fi.FiError, match="no CUDA device"):
        fi.SharedBuffer(1, 2)
    with pytest.raises(fi.FiError, match="no CUDA device"):
        fi.Learner(1, 4, 5, 2)


@pytest.mark.parametrize("s", [1, 4, 7])
def test_farmer_learner_rejects_trajectories_too_short_for_x(fi, s):
    """x[484] is carried in words 192..255 of records 0..7 (DESIGN.md, record layout): with fewer than 8 records a farmer
    learner would train on an x whose tail is zero. Creation refuses, before it looks for a device, so this runs anywhere."""
    with pytest.raises(fi.FiError, match=r"entry_size >= 8 \(x\[484\] spans records 0\.\.7\), got %d" % s):
        fi.Learner(1, 4, s, 2, model="farmer_lstm")


NAN, INF = float("nan"), float("inf")
VTRACE_REJECTED = ([(f, v) for f in ("rho_bar", "c_bar", "pg_rho_bar") for v in (NAN, 0.0, -0.5, -INF)] +
                   [("lambda_", v) for v in (NAN, -0.01, 1.01, INF, -INF)] +
                   [(f, v) for f in ("baseline_cost", "entropy_cost") for v in (NAN, -1e-3, INF, -INF)])


@pytest.mark.parametrize("field,value", VTRACE_REJECTED, ids=[f"{f}={v}" for f, v in VTRACE_REJECTED])
def test_actor_critic_learner_rejects_bad_vtrace_constants(fi, field, value):
    """A NaN clipping threshold would otherwise give NaN losses, and lambda outside [0, 1] or a negative loss weight a step
    that is not V-trace. Creation refuses with a message naming the field, before it looks for a device."""
    with pytest.raises(fi.FiError, match=rf"V-trace {field} must be .*, got"):
        fi.Learner(1, 4, 5, 2, model="mlp_actor_critic", **{field: value})


def test_unclipped_vtrace_constants_are_accepted(fi):
    """rho_bar = c_bar = pg_rho_bar = +inf means no clipping, with lambda and both costs at the ends of their ranges: creation
    gets past the configuration checks (without a device it then stops at the device lookup)."""
    import torch
    kw = dict(rho_bar=INF, c_bar=INF, pg_rho_bar=INF, lambda_=0.0, baseline_cost=0.0, entropy_cost=0.0)
    if torch.cuda.is_available():
        fi.Learner(1, 4, 5, 2, model="mlp_actor_critic", **kw).close()
        fi.Learner(1, 4, 5, 2, model="mlp_actor_critic", lambda_=1.0).close()
        return
    for k in (kw, dict(lambda_=1.0)):
        with pytest.raises(fi.FiError, match="no CUDA device"):
            fi.Learner(1, 4, 5, 2, model="mlp_actor_critic", **k)


def test_defaults_follow_the_reference_cli(fi):
    from freeimpala_b200 import _lib
    cfg = _lib.FiLearnerConfig()
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    # cmd/freeimpala/main.cpp:38-120 defaults: -p 2, -B 10, -S 100, -M 5; README bench lr 5e-4
    assert (cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size) == (2, 10, 100, 5)
    assert cfg.lr == 5e-4 and cfg.publish_every == 1


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under freeimpala_b200/ may reference it."""
    pkg = os.path.join(U.ROOT, "freeimpala_b200")
    for root, _, files in os.walk(pkg):
        if "_build" in root:
            continue
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".hpp", ".cpp")):
                text = open(os.path.join(root, f), errors="replace").read()
                assert "pyoracle" not in text and "liboracle" not in text and "oracle/" not in text, f


def test_reference_agent_header_compiles_against_the_host_shim(fi):
    """The reference's actor (include/freeimpala/agent.h), UNMODIFIED and compiled from where it lies, builds and links
    against freeimpala_b200/host/fi_host.hpp through the alias headers of oracle/ref_shim/dropin/ (INTEGRATION.md).
    Runs only where the reference tree is present; the resulting binary is exercised on the GPU by tests/test_gpu_host.py."""
    if not os.path.isdir("/root/reference/include/freeimpala"):
        pytest.skip("/root/reference is not present on this box")
    fi.load_library()
    from oracle import pyoracle as po
    subprocess.run(["make", "-C", os.path.join(U.ROOT, "oracle"), "-s", "dropin"], check=True)
    assert os.path.exists(po.DROPIN_BIN)
    # the alias headers define nothing of their own for the actor-private types: they re-export the reference's
    text = open(os.path.join(U.ROOT, "oracle", "ref_shim", "dropin", "freeimpala", "data_structures.h")).read()
    assert "using fi_reference::Buffer;" in text and "using SharedBuffer = fi_host::SharedBuffer;" in text
    # without a device the binary fails loudly (no CPU fallback)
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([po.DROPIN_BIN], capture_output=True, text=True)
        assert r.returncode != 0 and "no CUDA device" in r.stderr
