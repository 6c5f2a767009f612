"""The fused partition + exchange pass (mhb_partition_scatter_hist) on one GPU: the per-owner destinations all lie in
one local buffer, so what the multi-GPU build sends to other ranks' receive buffers can be checked directly."""
import ctypes as C

import numpy as np
import pytest

from megahit_b200 import lib

pytestmark = pytest.mark.gpu

TILE = {2: 6912, 3: 4608, 4: 3840, 5: 2304, 17: 768}  # records per tile of the pass at these widths


def _rows(x):
    """records as sortable opaque rows, so that two sets of records compare as multisets"""
    return np.sort(np.ascontiguousarray(x).view(np.dtype((np.void, x.shape[1] * 4))).reshape(-1))


@pytest.mark.parametrize("words", [2, 3, 4, 5, 17])
def test_partition_scatter_hist_fills_every_owner_region(words):
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    L = lib.load()
    world = 5
    n = 3 * TILE[words] + 17  # ragged last tile
    rng = np.random.default_rng(words)
    recs = rng.integers(0, 2 ** 32, size=(n, words), dtype=np.uint64).astype(np.uint32)
    byte = 4 * words - 1       # the leading byte: most significant byte of word 0
    next_byte = 4 * words - 2  # the byte each owner's sort visits first
    lead = recs[:, 0] >> 24
    nxt = (recs[:, 0] >> 16) & 255
    owner_of_byte = (np.arange(256) * world // 256).astype(np.uint8)
    owner = owner_of_byte[lead]
    count = np.bincount(owner, minlength=world)
    start = np.concatenate([[0], np.cumsum(count)])

    dev = torch.device("cuda")
    a = torch.from_numpy(recs.view(np.int32).reshape(-1).copy()).to(dev)
    slack = 64
    out = torch.full((n * words + slack,), -1, dtype=torch.int32, device=dev)
    addr = np.zeros(256, np.uint64)
    addr[:world] = out.data_ptr() + start[:world] * words * 4
    addr_dev = torch.from_numpy(addr.view(np.int64)).to(dev)
    lut_dev = torch.from_numpy(owner_of_byte).to(dev)
    ws = torch.zeros(L.mhb_sort_workspace_bytes(n, words), dtype=torch.uint8, device=dev)
    oh = torch.zeros(16 * 256, dtype=torch.int64, device=dev)
    done = C.c_int(0)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    lib._check(L.mhb_partition_scatter_hist(stream, C.c_void_p(a.data_ptr()), n, words, byte, C.c_void_p(lut_dev.data_ptr()),
                                            C.c_void_p(addr_dev.data_ptr()), C.c_void_p(ws.data_ptr()), ws.numel(), next_byte,
                                            C.c_void_p(oh.data_ptr()), C.byref(done)))
    torch.cuda.synchronize()
    assert done.value == 1

    got = out.cpu().numpy().view(np.uint32)
    assert (got[n * words:] == 0xFFFFFFFF).all(), "stores past the last owner region"
    got = got[: n * words].reshape(n, words)
    for o in range(world):
        region = got[start[o]:start[o + 1]]
        assert (_rows(region) == _rows(recs[owner == o])).all(), f"owner {o}: not a permutation of its records"

    exp_hist = np.zeros((16, 256), np.int64)
    np.add.at(exp_hist, (owner, nxt), 1)
    assert (oh.cpu().numpy().reshape(16, 256) == exp_hist).all()


def test_partition_scatter_needs_owner_table():
    """the exchange pass always partitions by owner: a NULL owner table is an argument error (checked before n)"""
    L = lib.load()
    assert L.mhb_partition_scatter(None, None, 0, 2, 7, None, None, None, 0) == 1  # MHB_ERR_ARG
