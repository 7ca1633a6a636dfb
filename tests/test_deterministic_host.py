"""CPU: the host side of the bit-reproducible native update -- `train --deterministic` sets training.cuda_deterministic, and
the workspace queries of the ordered GEMM / encoder gradient (pure host code: no GPU needed) size their partial buffers
with a slice count that depends on the problem alone."""
import pytest
import torch

from crowdnav_dsrnn_b200 import _lib, native
from crowdnav_dsrnn_b200 import train as train_mod


def test_deterministic_flag_sets_cuda_deterministic(monkeypatch):
    seen = []
    monkeypatch.setattr(train_mod, "train", lambda cfg, *a, **k: seen.append(cfg))
    train_mod.main(["--envs", "8", "--num_updates", "1", "--deterministic"])
    train_mod.main(["--envs", "8", "--num_updates", "1"])
    assert [c.training.cuda_deterministic for c in seen] == [True, False]


def _wgrad(rows, m, n, split):
    """dW = dY^T X problem (both operands MN-major) on host tensors: the query reads shapes only."""
    bf = lambda r, c: torch.zeros(r, c, dtype=torch.bfloat16)
    return dict(a=(bf(rows, m), bf(rows, m)), a_mn=True, b=(bf(rows, n), bf(rows, n)), b_mn=True,
                c=torch.zeros(m, n), split_k=split)


PROBLEMS = [(5000, 768, 256, 0), (5000, 768, 64, 0), (130, 384, 128, 1), (70000, 256, 512, 0), (999, 800, 72, 3),
            (2457600, 768, 256, 0), (2457600, 1024, 72, 0)]


def test_ordered_gemm_workspace_is_slices_times_m_n():
    for rows, m, n, split in PROBLEMS:
        nbytes, (s,) = native.ordered_workspace([_wgrad(rows, m, n, split)])
        kb = (rows + 63) // 64
        assert 1 <= s <= kb
        assert nbytes == (s * m * n * 4 if s > 1 else 0), (rows, m, n, split, s, nbytes)
    assert native.ordered_workspace([_wgrad(130, 384, 128, 1)])[1] == [1]
    assert native.ordered_workspace([_wgrad(999, 800, 72, 3)])[1] == [3]        # 16 k-blocks in 3 slices of 6, 6, 4
    assert native.ordered_workspace([_wgrad(999, 800, 72, 5)])[1] == [4]        # 5 slices of 4 would leave one empty: 4


def test_ordered_slice_count_does_not_depend_on_the_group():
    probs = [_wgrad(*p) for p in PROBLEMS]
    alone = [native.ordered_workspace([p]) for p in probs]
    for i in range(0, len(probs) - 3):
        group = probs[i:i + 4]
        nbytes, slices = native.ordered_workspace(group)
        assert slices == [a[1][0] for a in alone[i:i + 4]]
        assert nbytes == sum(a[0] for a in alone[i:i + 4])


def test_ordered_gemm_workspace_query_rejects_bad_problems():
    with pytest.raises(_lib.CrowdNavLibraryError):
        native.ordered_workspace([_wgrad(100, 64, 64, -1)])
    with pytest.raises(ValueError):
        native.ordered_workspace([_wgrad(100, 64, 64, 0)] * 5)


def test_encoder_grad_workspace_is_one_block_sum_per_block():
    lib = _lib.load()
    assert lib.cn_encoder_grad_ordered_workspace_bytes(0) == 0
    assert lib.cn_encoder_grad_ordered_workspace_bytes(5) == 2 * 192 * 4
    assert lib.cn_encoder_grad_ordered_workspace_bytes(30 * 4096 * 20) == 148 * 8 * 192 * 4


def test_ordered_predicate_defaults_off():
    assert native.DETERMINISTIC is False and not native.ordered()
