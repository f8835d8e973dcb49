"""CPU-only: the C-ABI library builds, loads and exports every symbol include/msw_b200.h
declares; the Python host mirror fails loudly without a GPU (no fallback)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from minesweeper_ppo_b200 import _lib, build
    build.build()
    return _lib.load()


def test_header_symbols_are_exported(lib):
    from minesweeper_ppo_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "msw_b200.h")).read()
    declared = set(re.findall(r"\b(msw_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in msw_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))


def test_binding_arity_matches_header():
    """ctypes silently accepts extra arguments and truncates them to 32 bits, so a binding that is
    one argtype short corrupts the last pointer (the stream).  Count the parameters of every
    prototype in the header and compare with the binding."""
    from minesweeper_ppo_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "msw_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    protos = dict(re.findall(r"\b(msw_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", hdr, flags=re.S))
    assert set(protos) == set(_lib.SIGNATURES)
    for name, params in protos.items():
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert n == len(_lib.SIGNATURES[name][1]), (name, n, len(_lib.SIGNATURES[name][1]))


def test_host_side_calls_without_device(lib):
    assert lib.msw_version() == 2
    assert lib.msw_words_per_board(16, 16) == 8 and lib.msw_words_per_board(16, 30) == 15
    assert lib.msw_words_per_board(32, 32) == 32 and lib.msw_words_per_board(33, 32) == 0
    assert lib.msw_words_per_board(16, 33) == 0


def test_no_cpu_fallback():
    import torch
    import minesweeper_ppo_b200 as m
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m.VecMinesweeper(4, m.EnvConfig())
    buf = m.RolloutBuffer(4, 2, (10, 8, 8), 64, torch.device("cpu"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        buf.compute_gae(torch.zeros(4))


def test_reward_constants_match_reference_bits():
    import numpy as np
    import minesweeper_ppo_b200 as m
    s, l, w = m.reward_constants(m.EnvConfig(H=16, W=16, mine_count=40, step_penalty=1e-4))
    assert [int(np.float32(x).view(np.uint32)) for x in (s, l, w)] == [0xB8D1B717, 0xBF800347, 0x3F7FF972]


def test_pack_boards_layout():
    import numpy as np
    import minesweeper_ppo_b200 as m
    b = np.zeros((2, 16 * 30), bool)
    b[0, 0] = b[0, 33] = b[1, 479] = True
    p = m.pack_boards(b, 480).view(np.uint32)
    assert p.shape == (2, 15) and p[0, 0] == 1 and p[0, 1] == 2 and p[1, 14] == 1 << 31


def test_product_never_imports_oracle():
    """The package must not import, link, load or call anything under oracle/."""
    pkg = os.path.join(ROOT, "minesweeper_ppo_b200")
    banned = re.compile(r"import\s+oracle|from\s+oracle|oracle\.|oracle/|libmsw_oracle|msw_oracle|\borc_[a-z]")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                hit = banned.search(open(os.path.join(dp, f)).read())
                assert hit is None, (f, hit.group(0))
