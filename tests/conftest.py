import os
import shutil
import sys
import tempfile

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# The trainers load CSVs through `datasets`, which caches under HF_HOME. Point the Hugging Face caches at a private
# directory for the session (set before any test module imports `datasets`), so the suite neither needs a writable
# user cache nor leaves anything in it; subprocesses started by tests inherit the setting.
_HF_TMP = tempfile.mkdtemp(prefix="dalm_b200_tests_hf_")
os.environ["HF_HOME"] = _HF_TMP
os.environ["HF_DATASETS_CACHE"] = os.path.join(_HF_TMP, "datasets")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (select with -m gpu)")


def pytest_unconfigure(config):
    shutil.rmtree(_HF_TMP, ignore_errors=True)


@pytest.fixture(scope="session")
def cuda_dev():
    import torch

    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from dalm_b200 import _lib

    _lib.call("dalm_b200_probe_device")
    return torch.device("cuda:0")
