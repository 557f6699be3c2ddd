"""The host side of the input gradients through the frozen predictor's shared windows: the reader CSRs (who reads each
row of the shared plan's pools, and which windows read each series row of the GRU's layer-0 projection) against a
brute-force transpose, and the routing of the residual builder."""
import pytest
import torch

from leak_det_gnn_b200.models import NormalPredictorTCN
from leak_det_gnn_b200.models.predictor import shared_cone_plan, shared_reader_plan, window_reader_csr

DIL = [1, 2, 4, 8]


def _brute(lists, ptr, idx):
    """The CSR (ptr, idx) equals the row lists ``lists`` exactly."""
    assert ptr.shape == (len(lists) + 1,) and int(ptr[0]) == 0
    assert torch.equal(ptr[1:] - ptr[:-1], torch.tensor([len(v) for v in lists], dtype=torch.int64))
    assert idx.tolist() == [m for v in lists for m in v]


def _transpose(src, n_rows):
    """Per tap and row r, the m with src[tap, m] == r in ascending m; row tap n_rows + r."""
    lists = [[] for _ in range(src.shape[0] * n_rows)]
    for tap, row in enumerate(src.tolist()):
        for m, r in enumerate(row):
            if r >= 0:
                lists[tap * n_rows + r].append(m)
    return lists


@pytest.mark.parametrize("window,length,count,batch", [(36, 72, 36, 2), (20, 41, 22, 3), (20, 41, 5, 2),
                                                       (64, 130, 67, 2), (64, 72, 9, 1), (36, 300, 200, 1)])
def test_tcn_reader_csrs_are_the_transposed_plan(window, length, count, batch):
    plan, _ = shared_cone_plan(length, window, count, batch, 3, DIL)
    readers = shared_reader_plan(plan, batch * length)
    n_in = batch * length
    for (src1, src2, res), (ptr1, idx1, ptr2, idx2, ptr_r, idx_r) in zip(plan, readers):
        _brute(_transpose(src1, n_in), ptr1, idx1)
        _brute(_transpose(src2, src1.shape[1]), ptr2, idx2)
        _brute(_transpose(res.view(1, -1), n_in), ptr_r, idx_r)
        # every (tap, m) with a source is listed exactly once; -1 (padding) never
        for src, idx in ((src1, idx1), (src2, idx2), (res.view(1, -1), idx_r)):
            assert idx.numel() == int((src >= 0).sum())
        n_in = res.numel()


def test_tcn_readers_are_not_injective():
    """A shared row near a window's left edge is read through one tap by several windows: the gather-form inverse of
    forward_cone cannot serve here."""
    plan, _ = shared_cone_plan(72, 36, 36, 1, 3, DIL)
    ptr1 = shared_reader_plan(plan, 72)[0][0]
    assert int((ptr1[1:] - ptr1[:-1]).max()) > 1


@pytest.mark.parametrize("length,window,count,batch", [(72, 36, 36, 2), (41, 20, 22, 3), (41, 20, 5, 2),
                                                       (130, 64, 67, 2), (36, 36, 1, 3)])
def test_gru_window_csr_is_the_transposed_gather(length, window, count, batch):
    ptr, idx = window_reader_csr(length, window, count, batch)
    lists = [[] for _ in range(batch * length)]
    for b in range(batch):
        for j in range(count):
            for p in range(window):
                lists[b * length + j + p].append((b * count + j) * window + p)
    _brute(lists, ptr, idx)
    assert idx.numel() == batch * count * window


def test_builder_without_gradients_on_the_cpu_is_unchanged():
    """Off the native path (CPU) the builder keeps the dense route and stays differentiable through plain autograd."""
    from leak_det_gnn_b200.models import build_residual_sequence_from_segment

    torch.manual_seed(0)
    m = NormalPredictorTCN(29, 9).eval().requires_grad_(False)
    noisy = torch.randn(2, 72, 29, requires_grad=True)
    tf = torch.randn(2, 72, 9)
    assert not m.differentiable_windows(noisy, tf)
    r = build_residual_sequence_from_segment(m, noisy, tf, 36, 36)
    r.sum().backward()
    assert noisy.grad is not None and noisy.grad.shape == noisy.shape
