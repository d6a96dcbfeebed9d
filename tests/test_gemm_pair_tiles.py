"""The fp16-pair tensor-core GEMM works on 256-row pair tiles (two CTAs, one M = 256 MMA).  Shapes whose 128-row tile
count is odd leave the last pair half empty; these cases run that over several waves of the resident pairs."""
import pytest
import torch

from spotv2net_b200._lib import check, ptr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

CASES = [
    # a_kc, b_kc, M, N, K, splits, bn (256 + 16: 32-element k-blocks), kb_per_chunk
    (1, 1, 4224, 3012, 1260, 1, 272, 0),     # 33 row tiles: 17 pair tiles x 12 column tiles, > 2 waves
    (0, 0, 3200, 1260, 8192, 4, 272, 0),     # 25 row tiles, split-K
    (1, 0, 4224, 1260, 3012, 1, 272, 0),
]


@pytest.mark.parametrize("case", CASES, ids=[f"{'KM'[c[0]]}{'KM'[c[1]]}_{c[2]}x{c[3]}x{c[4]}_s{c[5]}" for c in CASES])
def test_pair_tiles_with_odd_row_tile_count(cuda_lib, case):
    a_kc, b_kc, M, N, K, splits, bn, kbc = case
    torch.manual_seed(M + N + K)
    A = torch.randn(M, K) if a_kc else torch.randn(K, M)
    Bm = torch.randn(N, K) if b_kc else torch.randn(K, N)
    ref = (A.double() if a_kc else A.double().t()) @ (Bm.double() if b_kc else Bm.double().t()).t()
    Ag, Bg = A.to(DEV), Bm.to(DEV)
    ws = torch.empty(8 * (A.numel() + Bm.numel()) + 4 * splits * M * N + 8192, dtype=torch.uint8, device=DEV)
    Cg = torch.full((M, N), float("nan"), device=DEV)
    st = torch.cuda.current_stream().cuda_stream
    check(cuda_lib.spotv2_diag_gemm(a_kc, b_kc, M, N, K, ptr(Ag), A.shape[1], ptr(Bg), Bm.shape[1], ptr(Cg), N, 3, splits,
                                    bn, kbc, ptr(ws), ws.numel(), st), "diag_gemm fp16 pairs")
    torch.cuda.synchronize()
    err = ((Cg.double().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert err < 3e-6, err
