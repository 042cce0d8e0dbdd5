"""CPU checks of the layout-accuracy surface: IoU / mIoU / pixel accuracy derived from hand-built confusion counts, the
argument checks of vlg_confusion (no kernel is launched), and the data-parallel sum of the counts over two gloo ranks."""
import ctypes as C
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import vlg_b200
from vlg_b200 import _cabi, parallel


def _iou_with(conf, skipped=0):
    """LayoutIoU with one step whose counts are the given K x K matrix (on the CPU)."""
    conf = torch.as_tensor(conf, dtype=torch.int64)
    K = conf.shape[0]
    m = vlg_b200.LayoutIoU(n_classes=K, steps=1)
    m.counts[0, :K * K] = conf.reshape(-1)
    m.counts[0, K * K] = skipped
    return m


def test_perfect_prediction_gives_iou_one():
    r = _iou_with(torch.diag(torch.tensor([3, 1, 7, 2, 5]))).compute()
    assert torch.equal(r.iou, torch.ones(1, 5, dtype=torch.float64))
    assert r.miou.tolist() == [1.0] and r.pixel_acc.tolist() == [1.0]


def test_absent_class_is_nan_and_left_out_of_miou():
    # rows = target, columns = prediction; class 2 occurs in neither, class 4 is predicted but never a target
    conf = torch.tensor([[4, 1, 0, 0, 0],
                         [0, 3, 0, 0, 1],
                         [0, 0, 0, 0, 0],
                         [2, 0, 0, 6, 0],
                         [0, 0, 0, 0, 0]])
    r = _iou_with(conf).compute()
    want = [4 / (5 + 6 - 4), 3 / (4 + 4 - 3), math.nan, 6 / (8 + 6 - 6), 0 / (0 + 1 - 0)]
    got = r.iou[0].tolist()
    assert math.isnan(got[2])
    assert [g for i, g in enumerate(got) if i != 2] == pytest.approx([w for i, w in enumerate(want) if i != 2], abs=0)
    assert r.miou[0].item() == pytest.approx(sum(w for i, w in enumerate(want) if i != 2) / 4, abs=1e-15)
    assert r.pixel_acc[0].item() == pytest.approx(13 / 17, abs=1e-15)
    assert torch.equal(r.confusion[0], conf)


def test_pixel_accuracy_per_step():
    m = vlg_b200.LayoutIoU(n_classes=5, steps=3)
    m.counts[0, 0] = 10                       # all right
    m.counts[1, 0 * 5 + 1] = 4                # all wrong
    m.counts[1, 2 * 5 + 2] = 0
    m.counts[2, 3 * 5 + 3], m.counts[2, 3 * 5 + 4] = 3, 1
    r = m.compute()
    assert r.pixel_acc.tolist() == [1.0, 0.0, 0.75]
    assert r.iou.shape == (3, 5) and r.confusion.shape == (3, 5, 5)


def test_nothing_counted_gives_nan():
    r = vlg_b200.LayoutIoU(n_classes=5).compute()
    assert math.isnan(r.miou.item()) and math.isnan(r.pixel_acc.item())


def test_skipped_pixels_raise():
    m = _iou_with(torch.eye(5, dtype=torch.int64), skipped=3)
    with pytest.raises(vlg_b200.VlgError, match="outside"):
        m.compute()


def test_reset_and_sync_without_process_group():
    m = _iou_with(torch.eye(5, dtype=torch.int64) * 2)
    before = m.counts.clone()
    storage = m.counts.data_ptr()
    m.sync()                                  # identity without a process group
    assert torch.equal(m.counts, before)
    m.reset()
    assert m.counts.data_ptr() == storage and int(m.counts.abs().sum()) == 0
    assert torch.equal(parallel.sync_counts(before), before)


def test_step_out_of_range_is_refused():
    m = vlg_b200.LayoutIoU(n_classes=5, steps=2)
    lab = torch.zeros(1, 4, 4, dtype=torch.int64)
    with pytest.raises(vlg_b200.VlgError, match="step"):
        m.update(lab, lab, step=2)


def test_cpu_tensors_are_refused():
    lab = torch.zeros(1, 4, 4, dtype=torch.int64)
    with pytest.raises(vlg_b200.VlgError):
        vlg_b200.confusion_matrix(lab, lab, 5)


# ---------------------------------------------------------------- C ABI argument checks (nothing is launched)
FAKE = C.c_void_p(4096)   # never dereferenced: every call below is refused before a launch
ERR_ARG = -1              # VLG_ERR_ARG


def _confusion(prob, layout, pred, tgt, counts):
    lib = _cabi.load()
    return lib.vlg_confusion(C.byref(prob), layout, 0, pred, tgt, counts, None), lib.vlg_last_error()


def test_cabi_confusion_argument_checks():
    ok = _cabi.Problem(N=1, H=8, W=8, K=20)
    rc, err = _confusion(ok, FAKE, FAKE, FAKE, FAKE)
    assert rc == ERR_ARG and b"exactly one of layout / pred_label" in err
    rc, err = _confusion(ok, None, None, FAKE, FAKE)
    assert rc == ERR_ARG and b"exactly one of layout / pred_label" in err
    rc, err = _confusion(ok, None, FAKE, FAKE, None)
    assert rc == ERR_ARG and b"counts" in err
    rc, err = _confusion(ok, None, FAKE, None, FAKE)
    assert rc == ERR_ARG and b"tgt_label" in err
    rc, err = _confusion(_cabi.Problem(N=1, H=8, W=8, K=7), None, FAKE, FAKE, FAKE)
    assert rc != 0 and b"K=7" in err
    misaligned = C.c_void_p(4096 + 8)
    rc, err = _confusion(ok, misaligned, None, FAKE, FAKE)
    assert rc == ERR_ARG and b"16-byte aligned" in err
    rc, err = _confusion(_cabi.Problem(N=1, H=8, W=8, K=20, struct_size=96), None, FAKE, FAKE, FAKE)
    assert rc == ERR_ARG and b"struct_size" in err


# ---------------------------------------------------------------- two gloo ranks
K_DP = 19


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _labels(seed=7, N=6, H=9, W=11):
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, K_DP, (N, H, W), generator=g)
    t[torch.rand(N, H, W, generator=g) < 0.1] = -100
    p = torch.randint(0, K_DP, (N, H, W), generator=g)
    return p, t


def _oracle_counts(p, t, K=K_DP, ignore=-100):
    keep = t != ignore
    out = torch.zeros(K * K + 1, dtype=torch.int64)
    out[:K * K] = torch.bincount((t * K + p)[keep], minlength=K * K)
    return out


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    p, t = _labels()
    lo, hi = parallel.shard_bounds(p.shape[0], rank, world)
    local = torch.stack([_oracle_counts(p[lo:hi], t[lo:hi]), _oracle_counts(p[lo:hi].flip(0), t[lo:hi])])
    reduced = parallel.sync_counts(local)
    m = vlg_b200.LayoutIoU(n_classes=K_DP, steps=2)
    m.counts.copy_(local)
    m.sync()
    if rank == 0:
        q.put((reduced.numpy(), m.counts.numpy()))
    dist.destroy_process_group()


def test_two_rank_counts_match_single_process():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    reduced, synced = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    p, t = _labels()
    flipped = torch.cat([p[0:3].flip(0), p[3:6].flip(0)])   # the shards of rank 0 and 1, each flipped on its own
    full = torch.stack([_oracle_counts(p, t), _oracle_counts(flipped, t)]).numpy()
    assert (reduced == full).all() and reduced.dtype == full.dtype
    assert (synced == full).all()
