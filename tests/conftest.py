import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLD = ROOT / "tests" / "golden"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


# `-m gpu` tests on a box without a GPU fail loudly (QlbError from Context): the product has no CPU path to skip to.


@pytest.fixture(scope="session")
def oracle():
    from oracle.bindings import Restatement
    return Restatement()


@pytest.fixture(scope="session")
def matrices():
    from qkd_ldpc_b200 import codes
    return {p.stem: codes.load_npz(p) for p in sorted(codes.CODES.glob("*.npz"))}


@pytest.fixture(scope="session")
def graphs(matrices):
    from oracle.bindings import Graph
    return {k: Graph(m.n, m.m, m.row_ptr, m.col_idx, m.col_ptr, m.row_idx, is_regular=m.is_regular, max_bit_w=m.max_bit_w,
                     max_check_w=m.max_check_w) for k, m in matrices.items()}


@pytest.fixture(scope="session")
def lib():
    from qkd_ldpc_b200 import capi
    return capi.load_library()


@pytest.fixture(scope="session")
def ctx(lib):
    from qkd_ldpc_b200 import capi
    return capi.Context(0)


@pytest.fixture(scope="session")
def dev_codes(matrices):
    from qkd_ldpc_b200 import capi
    return {k: capi.Code.from_graph(m) for k, m in matrices.items()}


NS = "n10240_m5231_cw3_seed666"
