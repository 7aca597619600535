"""The per-block comparator of the GPU parity tests (tests/gpu_bringup.py:_metrics) on CPU tensors.

The GEMM kernels fail locally: an epilogue skipped on the rows of the partial last row tile, a k-block lost in one
stream-K hand-over.  At 9625 x 512 x 2048 (a tower shape the GPU suite runs with every epilogue) such a fault is diluted
below the whole-tensor bf16 bound by the correct rest of the output.  These tests emulate the faults on a correctly
rounded bf16 output and check that the per-tile metric rejects them while it accepts the correct output."""
import pytest
import torch

from tests import gpu_bringup as gb
from tests.test_gpu_parity import BF16_REL

M, N, K = 9625, 512, 2048  # 75 full 128-row tiles + a 25-row tail


@pytest.fixture(scope="module")
def gemm_case():
    g = torch.Generator().manual_seed(0)
    A = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    B = (torch.randn(N, K, generator=g) * 0.5).bfloat16()
    bias = torch.randn(N, generator=g)
    prod = A.double() @ B.double().t()
    ref = prod + bias.double()
    good = ref.bfloat16()
    # bias dropped on the rows of the partial last row tile (an M-tail epilogue bug)
    tail0 = M // 128 * 128
    tail = good.clone()
    tail[tail0:] = prod[tail0:].bfloat16()
    # one 64-wide k-block missing in one 128 x 256 tile (a lost stream-K hand-over)
    r0, c0, k0 = 3 * 128, 256, 17 * 64
    kblk = good.clone()
    lost = A[r0:r0 + 128, k0:k0 + 64].double() @ B[c0:c0 + 256, k0:k0 + 64].double().t()
    kblk[r0:r0 + 128, c0:c0 + 256] = (ref[r0:r0 + 128, c0:c0 + 256] - lost).bfloat16()
    return {"A": A, "B": B, "bias": bias, "ref": ref, "good": good, "tail": tail, "kblk": kblk, "tail0": tail0,
            "kblk_tile": [r0, c0]}


def test_block_metric_accepts_correct_bf16_output(gemm_case):
    m = gb._metrics(gemm_case["good"], gemm_case["ref"], tile=gb.GEMM_TILE)
    assert m["blk_rel"] <= BF16_REL and m["rel"] <= BF16_REL, m
    e = gb._gemm_elementwise(gemm_case["good"], gemm_case["ref"], gemm_case["A"], gemm_case["B"], "bf16", bias=gemm_case["bias"])
    assert e["elem_ratio"] <= 1.0, e


def test_whole_tensor_metric_misses_bias_dropped_on_the_m_tail(gemm_case):
    """The reason for the block metric: the old whole-tensor rel-L2 accepts this fault."""
    assert gb._metrics(gemm_case["tail"], gemm_case["ref"])["rel"] <= BF16_REL


def test_block_metric_rejects_bias_dropped_on_the_m_tail(gemm_case):
    m = gb._metrics(gemm_case["tail"], gemm_case["ref"], tile=gb.GEMM_TILE)
    assert m["blk_rel"] > 10 * BF16_REL, m
    assert m["blk_worst"][0] == gemm_case["tail0"], m  # the failure names a tile of the tail
    e = gb._gemm_elementwise(gemm_case["tail"], gemm_case["ref"], gemm_case["A"], gemm_case["B"], "bf16", bias=gemm_case["bias"])
    assert e["elem_ratio"] > 1.0 and e["elem_worst"][0] >= gemm_case["tail0"], e


def test_block_metric_rejects_one_missing_k_block(gemm_case):
    m = gb._metrics(gemm_case["kblk"], gemm_case["ref"], tile=gb.GEMM_TILE)
    assert m["blk_rel"] > 10 * BF16_REL, m
    r0, c0 = gemm_case["kblk_tile"]
    assert r0 <= m["blk_worst"][0] < r0 + 128 and c0 <= m["blk_worst"][1] < c0 + 256, m


def test_block_metric_grid_layout_and_near_zero_blocks():
    """grid= names the worst block by its index; a block whose reference is ~0 is judged against the floor, not
    against its own (vanishing) norm, so rounding noise there cannot fail it, while a real error there still does."""
    g = torch.Generator().manual_seed(1)
    S, H, L = 3, 4, 16
    ref = torch.randn(S, H, L * 64, generator=g, dtype=torch.float64)
    ref[1, 2] *= 1e-9  # a (sequence, head) problem with a near-zero reference
    noisy = ref * (1 + 1e-3 * torch.randn(ref.shape, generator=g, dtype=torch.float64))
    noisy[1, 2] += 1e-4 * torch.randn(L * 64, generator=g, dtype=torch.float64)  # rounding noise at the tensor's scale
    m = gb._metrics(noisy, ref, grid=(S, H))
    assert m["blk_rel"] < 2e-3, m
    bad = noisy.clone()
    bad[2, 1, :64] += 0.5  # one query row of one problem wrong
    m = gb._metrics(bad, ref, grid=(S, H))
    assert m["blk_rel"] > 0.05 and m["blk_worst"] == [2, 1], m
    unwritten = ref.clone()
    unwritten[0, 3, 5] = float("nan")
    m = gb._metrics(unwritten, ref, grid=(S, H))
    assert m["blk_rel"] == float("inf") and m["blk_worst"] == [0, 3], m
