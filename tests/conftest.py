import os
import subprocess
import sys

# The checker (numpy oracle: thousands of small matmuls; C restatement: OpenMP) must not fan out over every logical CPU of a
# 128-thread GPU box: BLAS / OpenMP thread pools that large spend their time synchronising, and the round-2 GPU suite took 21
# minutes (331 CPU-minutes) instead of two.  Set BEFORE numpy loads its BLAS.  bench.py is not affected (it picks the CPU
# baseline's thread count itself).
for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, str(max(1, min(16, (os.cpu_count() or 8)))))

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


try:        # numpy may have been imported by a plugin before this file ran: cap the pools that already exist as well
    from threadpoolctl import threadpool_limits
    threadpool_limits(limits=int(os.environ["OPENBLAS_NUM_THREADS"]))
except Exception:
    pass


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def tmp_models(tmp_path_factory):
    return tmp_path_factory.mktemp("models")


@pytest.fixture(scope="session")
def tiny_gguf(tmp_models):
    """2-layer d=256 Llama (head_dim 64, GQA 2:1), q4_K_M recipe (Q4_K + Q6_K), properly quantised."""
    from oracle import gguf_synth as S
    p = str(tmp_models / "tiny_q4km.gguf")
    S.build_model(p, S.TINY, "q4_k_m", seed=1234)
    return p


@pytest.fixture(scope="session")
def tiny128_gguf(tmp_models):
    """2-layer d=512 Llama with head_dim 128, GQA 4:1, n_ff 768, q4_K_M recipe."""
    from oracle import gguf_synth as S
    p = str(tmp_models / "tiny128_q4km.gguf")
    S.build_model(p, S.TINY128, "q4_k_m", seed=4321)
    return p


@pytest.fixture(scope="session")
def mid_gguf(tmp_models):
    """2-layer d=1024 Llama (head_dim 128, GQA 4:1, n_ff 2048): wide enough for the cluster path of the batched GEMMs."""
    from oracle import gguf_synth as S
    p = str(tmp_models / "mid_q4km.gguf")
    S.build_model(p, S.MID, "q4_k_m", seed=2468)
    return p


@pytest.fixture(scope="session")
def tiny_q8_gguf(tmp_models):
    from oracle import gguf_synth as S
    p = str(tmp_models / "tiny_q8.gguf")
    S.build_model(p, S.TINY, "q8_0", seed=99)
    return p


@pytest.fixture(scope="session")
def tiny_f16_gguf(tmp_models):
    from oracle import gguf_synth as S
    p = str(tmp_models / "tiny_f16.gguf")
    S.build_model(p, S.TINY, "f16", seed=77)
    return p


@pytest.fixture(scope="session")
def hostcheck_lib(tmp_path_factory):
    """CPU build of the GEMV lane program (tests/hostcheck) -- test infrastructure only.  Built afresh every session, outside
    the tree, so it always matches the product headers it includes."""
    import ctypes
    src = os.path.join(ROOT, "tests", "hostcheck", "hostcheck.cpp")
    out = str(tmp_path_factory.mktemp("hostcheck") / "libhostcheck.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", out, src,
                           os.path.join(ROOT, "gridllm_b200", "csrc", "gguf_file.cpp"),
                           os.path.join(ROOT, "gridllm_b200", "csrc", "tokenizer.cpp")])
    return ctypes.CDLL(out)


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))
