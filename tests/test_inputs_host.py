"""The rule for device frames the GMM and DTW entry points accept (``mixture.device_frames``), on CPU-built inputs: every
refusal branch raises ``ValueError`` before anything reaches a device, and the accepted forms come back with int64
offsets.  No GPU needed: the helper compares devices without touching one."""
import numpy as np
import pytest
import torch

from speech_signal_processing_b200.mixture import device_frames

DEV = torch.device("cuda:0")


def meta(rows, cols, dtype=torch.float32):
    """A tensor that claims to be on cuda:0 without one: the meta device's tensors carry shape, dtype and strides only."""
    return torch.empty((rows, cols), dtype=dtype, device="meta")


def test_a_cpu_tensor_is_refused_whatever_its_form():
    x = torch.zeros((6, 3))
    with pytest.raises(ValueError, match="is on cpu"):
        device_frames(x, [0, 6], DEV)


def test_the_device_must_be_the_set_s_device():
    x = torch.zeros((6, 3))
    with pytest.raises(ValueError, match="cuda:1"):
        device_frames(x, [0, 6], torch.device("cuda:1"))
    with pytest.raises(ValueError, match="is on meta"):
        device_frames(meta(6, 3), [0, 6], DEV)


@pytest.mark.parametrize("dtype", [torch.float64, torch.float16, torch.bfloat16, torch.int32])
def test_every_dtype_but_float32_is_refused(dtype):
    with pytest.raises(ValueError, match="float32"):
        device_frames(torch.zeros((6, 3), dtype=dtype), [0, 6], torch.device("cpu"))


@pytest.mark.parametrize("shape", [(6,), (2, 3, 1), ()])
def test_only_2d_tensors(shape):
    with pytest.raises(ValueError, match="2-D"):
        device_frames(torch.zeros(shape), [0, 1], torch.device("cpu"))


def test_numpy_and_lists_are_not_device_tensors():
    with pytest.raises(ValueError, match="torch tensor"):
        device_frames(np.zeros((6, 3), dtype=np.float32), [0, 6], torch.device("cpu"))


def test_strided_views_are_refused_and_row_ranges_accepted():
    cpu = torch.device("cpu")
    wide = torch.zeros((8, 40))
    with pytest.raises(ValueError, match="contiguous"):
        device_frames(wide[:, :39], [0, 8], cpu)                 # column slice: rows 40 floats apart
    with pytest.raises(ValueError, match="contiguous"):
        device_frames(wide[:, :1], [0, 8], cpu)                  # one column of it
    with pytest.raises(ValueError, match="contiguous"):
        device_frames(torch.zeros((39, 8)).T, [0, 8], cpu)       # y.T of a (D, T) matrix
    with pytest.raises(ValueError, match="contiguous"):
        device_frames(wide[::2], [0, 4], cpu)                    # every other row
    big = torch.zeros((9, 40))
    got = device_frames(big[1:], np.array([0, 3, 8], dtype=np.int32), cpu)   # row range: 4 bytes past the base
    assert got.dtype == np.int64 and got.tolist() == [0, 3, 8]
    assert device_frames(wide[2:2], [0], cpu).tolist() == [0]                # no rows, no utterances
    assert device_frames(wide[:1, :39], [0, 1], cpu).tolist() == [0, 1]      # one row of a column slice is contiguous


@pytest.mark.parametrize("offsets, why", [
    ([0, 3, 2, 6], "decrease"),
    ([1, 3, 6], "start above 0"),
    ([-1, 3, 6], "start below 0"),
    ([0, 3, 7], "end beyond the rows"),
    ([0, 3, 5], "end before the rows"),
    ([0, 3.0, 6], "float offsets"),
    ([[0, 6]], "2-D offsets"),
    ([], "no offsets"),
    ([False, True], "boolean offsets"),
])
def test_offsets_refusals(offsets, why):
    with pytest.raises(ValueError, match="offsets"):
        device_frames(torch.zeros((6, 3)), offsets, torch.device("cpu"))


def test_empty_utterances_are_accepted():
    """The GMM kernels score utterances of 0 frames (their score is 0); DTW adds its own rule on top."""
    got = device_frames(torch.zeros((6, 3)), np.array([0, 0, 6, 6], dtype=np.uint32), torch.device("cpu"))
    assert got.dtype == np.int64 and got.tolist() == [0, 0, 6, 6]


def test_the_check_reads_no_device():
    """Offsets come from the host and the tensor is only inspected: a meta tensor (no storage at all) passes the rule
    once the device matches."""
    assert device_frames(meta(6, 3), [0, 2, 6], torch.device("meta")).tolist() == [0, 2, 6]
