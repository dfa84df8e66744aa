"""Host-only checks of the markers-only forward pass: the facade binary builds with plain g++ over the C ABI."""
import os

from test_task_forward_gpu import _build_facade


def test_cpp_facade_task_forward_builds_without_cuda_headers(tmp_path):
    """tests/cpp/facade_task_forward.cpp (smplpp::IkTaskSet::calcActualPositions) compiles and links with g++ alone."""
    assert os.path.exists(_build_facade(tmp_path))
