"""The tcgen05 "rows" product on an A taller than 2^31 rows.

The tensor map that feeds A to the kernel takes 32-bit row coordinates, so a taller A runs in chunks of 2^31 - 128
rows, each with a map of its own.  A row's result must not depend on the chunk it lands in.  The entries are small
integers, so every 3xTF32 partial sum is exact and the fp64 product cast to fp32 is the only correct answer.  A and C
take 32 GiB each.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

M = (1 << 31) + 256
CHUNK = (1 << 31) - 128


def test_rows_product_is_exact_across_the_row_chunks():
    import pygcn_b200 as P

    assert P._lib.load().gcnb_check_device() == 0, P._lib.last_error()
    dev = torch.device("cuda:0")
    gen = torch.Generator(device=dev).manual_seed(0)
    a = torch.randint(-8, 9, (M, 4), generator=gen, device=dev, dtype=torch.float32)
    b = torch.randint(-8, 9, (4, 4), generator=gen, device=dev, dtype=torch.float32)
    try:
        c = P.mm(a, b, precision="tf32x3")
        for rows in (slice(0, 256), slice(CHUNK - 128, CHUNK + 128), slice(M - 256, M)):
            ref = (a[rows].double() @ b.double()).float()
            assert torch.equal(c[rows], ref), rows
    finally:
        a = c = None
        torch.cuda.empty_cache()
