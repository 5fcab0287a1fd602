"""CPU: the C-ABI library loads and exports every symbol include/gcrl_b200.h declares;
host-side logic that needs no GPU (LR schedule, error mapping, no-CPU-fallback rule)."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gcrl_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gcrl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from gcrl_b200 import _lib
    dll = ctypes.CDLL(_lib.library_path())
    names = declared_symbols()
    assert len(names) >= 35
    for n in names:
        assert hasattr(dll, n), f"{n} declared in include/gcrl_b200.h but not exported"
    # and the Python binding binds exactly the declared set
    assert sorted(_lib.SIGNATURES) == names


def test_abi_version_and_error_string():
    from gcrl_b200 import _lib
    assert _lib.lib.gcrl_abi_version() == 5
    assert isinstance(_lib.lib.gcrl_last_error(), bytes)


def test_agent_config_struct_matches_header():
    from gcrl_b200._lib import AgentConfig
    src = open(HEADER).read()
    body = re.search(r"typedef struct gcrl_agent_config \{(.*?)\} gcrl_agent_config;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"(?:int32_t|float)\s+([a-z_0-9]+)\s*;", body)
    assert fields == [f[0] for f in AgentConfig._fields_]
    assert ctypes.sizeof(AgentConfig) == 4 * len(fields)


def test_sac_config_struct_matches_header():
    from gcrl_b200._lib import SacConfig
    src = open(HEADER).read()
    body = re.search(r"typedef struct gcrl_sac_config \{(.*?)\} gcrl_sac_config;", src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = []
    for decl in re.findall(r"(?:int32_t|float)\s+([a-z_0-9, ]+);", body):
        fields += [f.strip() for f in decl.split(",")]
    assert fields == [f[0] for f in SacConfig._fields_]
    assert ctypes.sizeof(SacConfig) == 4 * len(fields)


def test_header_compiles_as_plain_c_and_struct_sizes_agree(tmp_path):
    """The boundary is a C ABI: the header must be consumable by a C compiler (no C++ in the signatures), and the
    structs the Python binding mirrors must have the sizes the C compiler gives them."""
    import shutil
    import subprocess
    from gcrl_b200._lib import AgentConfig, SacConfig
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "abi.c"
    src.write_text('#include <stdio.h>\n#include "gcrl_b200.h"\n'
                   'int main(void) { printf("%zu %zu %d\\n", sizeof(gcrl_agent_config), sizeof(gcrl_sac_config), '
                   'GCRL_ABI_VERSION); return 0; }\n')
    exe = tmp_path / "abi"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(src), "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert [int(x) for x in out] == [ctypes.sizeof(AgentConfig), ctypes.sizeof(SacConfig), 5]


def test_quantile_critic_loss_refuses_bad_arguments():
    """gcrl_quantile_critic_loss checks its sizes, leading dimensions and operands before it touches a device (every
    buffer is NULL: nothing here can launch)."""
    from gcrl_b200._lib import ERR_INVALID, lib

    def call(n=5, M=25, drop=2, B=64, ldm=28, zstride=64 * 28, ldy=116, coef=0.2):
        return lib.gcrl_quantile_critic_loss(0, n, M, drop, B, None, None, ldm, zstride, None, None, None, None, 0.98,
                                             coef, None, None, ldy, None, None, None, None, None)
    for kw, msg in [(dict(n=0), b"n_critics"), (dict(n=9), b"n_critics"), (dict(M=0), b"n_quantiles"),
                    (dict(n=8, M=33, ldm=36, zstride=64 * 36), b"256"), (dict(drop=25), b"drop"),
                    (dict(drop=-1), b"drop"), (dict(B=0), b"batch"), (dict(ldm=24), b"ldm"), (dict(ldm=30), b"ldm"),
                    (dict(zstride=64 * 28 - 1), b"zstride"), (dict(ldy=112), b"ldy"), (dict(ldy=118), b"ldy"),
                    (dict(coef=-1.0), b"alpha_dev"), ({}, b"NULL")]:
        assert call(**kw) == ERR_INVALID, kw
        assert msg in lib.gcrl_last_error(), (kw, lib.gcrl_last_error())


def test_no_cpu_fallback_without_device():
    """Without a GPU the product must fail loudly, never compute on the host."""
    from gcrl_b200 import _lib
    if _lib.device_count() > 0:
        pytest.skip("GPU present")
    from gcrl_b200 import HERBuffer, PERBuffer, ReplayBuffer, RunningNormalizer
    with pytest.raises(_lib.GcrlError):
        HERBuffer(1000, 50, 1)
    with pytest.raises(_lib.GcrlError):
        RunningNormalizer(3)
    with pytest.raises(_lib.GcrlError):
        PERBuffer(1000, 0.6)
    with pytest.raises(_lib.GcrlError):
        ReplayBuffer(1000)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "goal-conditioned-rl-framework_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("# oracle-free", ""), os.path.join(dirpath, f)


def test_cosine_schedule_matches_torch():
    import torch
    from gcrl_b200 import CosineAnnealingLR
    for base, T, eta in ((1e-3, 1, 1e-3), (1e-3, 3, 1e-4), (2e-3, 2, 5e-4), (5e-4, 7, 1e-5)):
        p = torch.nn.Parameter(torch.zeros(1))
        opt = torch.optim.SGD([p], lr=base)
        ref = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=T, eta_min=eta)
        mine = CosineAnnealingLR(base, T, eta)
        for _ in range(25):
            opt.step()
            ref.step()
            mine.step()
            assert math.isclose(mine.lr, opt.param_groups[0]["lr"], rel_tol=1e-12, abs_tol=1e-18)


def test_oracle_feistel_restatement_is_a_permutation():
    from oracle.index_stream import feistel_positions
    for n in (1, 2, 3, 7, 64, 777, 4097):
        for epoch in (0, 1, 5):
            p = feistel_positions(np.arange(n), n, seed=1898, epoch=epoch)
            assert sorted(p.tolist()) == list(range(n))
    a = feistel_positions(np.arange(256), 100000, 1898, 0)
    b = feistel_positions(np.arange(256), 100000, 1898, 1)
    assert len(set(a.tolist())) == 256 and not np.array_equal(a, b)
