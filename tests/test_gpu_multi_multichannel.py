"""2-GPU test of the distributed drivers with a 3-channel image (skipped with fewer than 2 GPUs): the latency mode
(infer_volume_distributed, with and without roi padding) and the throughput mode (infer_volumes_distributed over both
exchanges) give the labels of single-GPU infer_volume."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.util import SMALL, seeded_image, seeded_noise

pytestmark = pytest.mark.gpu

K = 3  # image channels


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _image(shape, seed):
    return torch.cat([seeded_image((1, 1) + tuple(shape), seed=seed + 10 * c) for c in range(K)], 1)


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import diff_unet_amos_b200 as pkg

    cout, S = 4, 32
    torch.manual_seed(0)
    m = pkg.DiffUNetB200(in_channels=K, out_channels=cout, image_size=S, spatial_size=S, features=SMALL).cuda().eval()
    # (48, 56, 40): plain case.  (48, 56, 24): one axis smaller than the roi -> the driver pads and must crop back
    for tag, vol in (("", (48, 56, 40)), ("_padded", (48, 56, 24))):
        image = _image(vol, 1).cuda()
        padded = tuple(max(v, S) for v in vol)
        n_win = len(pkg.window_starts(padded, (S, S, S), 0.25))
        noise = seeded_noise((n_win, cout, S, S, S)).cuda()
        nf = lambda w, b: noise[w:w + b]
        blended, labels = pkg.infer_volume_distributed(m, image, sw_batch_size=2, overlap=0.25, noise_fn=nf)
        if rank == 0:
            ref_b, ref_l = pkg.infer_volume(m, image, sw_batch_size=2, overlap=0.25, noise_fn=nf)
            ret["rel" + tag] = float((blended - ref_b).norm() / ref_b.norm())
            ret["equal" + tag] = bool(torch.equal(labels, ref_l))
            ret["shape_ok" + tag] = tuple(blended.shape) == tuple(ref_b.shape) == (1, cout) + vol
        else:
            assert blended is None and labels is None
    # throughput mode: three volumes as window queues, library noise keyed by (seed, global window index)
    vol = (48, 56, 40)
    images = [_image(vol, 20 + i).cuda() for i in range(3)]
    n_win = len(pkg.window_starts(vol, (S, S, S), 0.25))
    st = pkg.window_starts(vol, (S, S, S), 0.25)
    refs = []
    if rank == 0:
        for i, img in enumerate(images):
            b = pkg.StitchBuffers(cout, vol, (S, S, S), 0.25, "cuda")
            for g in range(0, n_win, 2):
                b.add_windows(m, img[0], st[g:g + 2], seed=11, noise_ids=range(i * n_win + g, i * n_win + min(g + 2, n_win)))
            refs.append(b.finalize(binary=True)[1])
    for exchange in ("p2p", "nccl"):
        outs = pkg.infer_volumes_distributed(m, images, sw_batch_size=2, overlap=0.25, seed=11, exchange=exchange)
        if rank == 0:
            ret["queue_n_" + exchange] = len(outs)
            ret["queue_equal_" + exchange] = all(bool(torch.equal(o, r)) for o, r in zip(outs, refs))
        else:
            assert outs is None
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_three_channel_volume_equals_single_gpu():
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(2, _free_port(), ret), nprocs=2, join=True)
    print("2-GPU 3-channel check:", dict(ret))
    for tag in ("", "_padded"):
        assert ret["shape_ok" + tag], tag
        assert ret["rel" + tag] < 1e-6 and ret["equal" + tag], tag  # fp32 sums in a different order only
    for exchange in ("p2p", "nccl"):
        assert ret["queue_n_" + exchange] == 3 and ret["queue_equal_" + exchange], exchange
