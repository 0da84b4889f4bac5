"""GPU, >= 2 devices (skipped on a 1-GPU box): BASELINE configs 4 and 5 over NCCL / NVLink, checked
against the CPU ORACLE (not against a 1-GPU run of the same kernels).
config 5: one long stream split into time segments; the (ntaps-1)-sample halo is read in place from the
left neighbour's buffer (PeerHalo: CUDA IPC + peer access) and, as the portable form, exchanged
point-to-point; NCCL gather of the outputs == oracle.fir of the whole stream.
config 4: channelizer, both partitions of SURVEY.md 8(e): output channels sharded per GPU == the
columns of oracle.pfb_channelizer; time segments with a (P-1)*M-sample halo == its rows."""
import os
import socket

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import scipy.signal as sig
    import newsched_b200 as nb
    import oracle as o
    from newsched_b200 import multigpu as mg
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ok, notes = True, []
    try:
        rng = np.random.default_rng(11)
        n_all = 1 << 20
        x_all = (rng.uniform(-1, 1, n_all) + 1j * rng.uniform(-1, 1, n_all)).astype(np.complex64)
        for T, D, algo, n in ((64, 1, 1, 1 << 20), (4096, 1, 3, 1 << 18), (1024, 4, 0, 1 << 20), (256, 1, 2, 1 << 20)):
            x = x_all[:n]
            taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
            lo, hi = mg.time_segments(n, world, D, halo_len=T - 1)[rank]
            seg = torch.from_numpy(x[lo:hi]).cuda()
            ref = o.fir(x, taps, D) if rank == 0 else None
            for peer in (True, False):
                fir = nb.FirFilter(taps, D, algorithm=algo)
                y = mg.SegmentedFir(fir, rank, world, peer=peer).run(seg)
                full = mg.gather_concat(y, rank, world)
                if rank == 0:
                    err = o.rel_rms(full.cpu().numpy(), ref)
                    good = full.numel() == ref.size and err < 1e-5
                    notes.append((T, D, fir.algorithm, "peer" if peer else "p2p", float(err)))
                    ok &= bool(good)
                    if algo == 1:      # direct form: bit-identical to the single stream
                        one = nb.FirFilter(taps, D, algorithm=1).work(torch.from_numpy(x).cuda())[0]
                        ok &= bool(torch.equal(full, one))
        # config 4
        M, P = 64, 16
        pt = sig.firwin(M * P, 1.0 / M).astype(np.float32)
        nx = M * 8192
        x = x_all[:nx]
        refc = o.pfb_channelizer(x, pt, M) if rank == 0 else None          # [frames, M]
        # (a) channels sharded, every GPU reads the whole stream
        xs = torch.from_numpy(x).cuda()
        b, c = mg.channel_slice(M, rank, world)
        part = nb.PfbChannelizer(pt, M, channel_begin=b, channel_count=c).work(xs)[0]
        cols = mg.gather_concat(part.t().contiguous(), rank, world)       # gather along channels
        if rank == 0:
            err = o.rel_rms(cols.t().cpu().numpy().reshape(-1), refc.reshape(-1))
            notes.append(("pfb", "channels", float(err)))
            ok &= bool(err < 1e-5)
        # (b) time segments, (P-1)*M halo read from the neighbour in place
        lo, hi = mg.time_segments(nx, world, M, halo_len=(P - 1) * M)[rank]
        seg = torch.from_numpy(x[lo:hi]).cuda()
        pfb = nb.PfbChannelizer(pt, M)
        for peer in (True, False):
            rows = mg.SegmentedFir(pfb, rank, world, peer=peer, halo_len=(P - 1) * M).run(seg)
            allrows = mg.gather_concat(rows.contiguous(), rank, world)
            if rank == 0:
                err = o.rel_rms(allrows.cpu().numpy().reshape(-1), refc.reshape(-1))
                notes.append(("pfb", "time", "peer" if peer else "p2p", float(err)))
                ok &= bool(err < 1e-5)
        torch.cuda.synchronize()
        if rank == 0:
            q.put((ok, notes))
    finally:
        dist.destroy_process_group()


def test_configs_4_and_5_on_two_gpus_match_the_oracle():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    ok, notes = q.get(timeout=5)
    assert ok is True, notes


# ---- the same sharding logic on ONE GPU: two ranks (processes) share cuda:0, host plumbing over gloo, the halo
# read in place through the CUDA IPC mapping -- so the driver's 1-GPU box exercises configs 4 / 5 at N = 2 too
def _worker_one_gpu(rank, world, port, q):
    import torch
    import torch.distributed as dist
    import scipy.signal as sig
    import newsched_b200 as nb
    import oracle as o
    from newsched_b200 import multigpu as mg
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ok, notes = True, []

    def gather_cpu(t):
        parts = [None] * world
        dist.all_gather_object(parts, t.cpu().numpy())
        return np.concatenate(parts)

    try:
        rng = np.random.default_rng(13)
        n = 1 << 19
        x = (rng.uniform(-1, 1, n) + 1j * rng.uniform(-1, 1, n)).astype(np.complex64)
        for T, D, algo in ((64, 1, 1), (128, 1, 2), (4096, 1, 3), (1024, 4, 0)):
            taps = (rng.uniform(-1, 1, T) / T).astype(np.float32)
            lo, hi = mg.time_segments(n, world, D, halo_len=T - 1)[rank]
            seg = torch.from_numpy(x[lo:hi]).cuda()
            fir = nb.FirFilter(taps, D, algorithm=algo)
            sf = mg.SegmentedFir(fir, rank, world, peer=True)
            y = sf.run(seg)
            torch.cuda.synchronize()
            full = gather_cpu(y)
            err = o.rel_rms(full, o.fir(x, taps, D, mt=True))
            notes.append((T, D, fir.algorithm, float(err)))
            ok &= bool(err < 1e-5)
            dist.barrier()          # nobody unmaps / frees while the neighbour may still read
            sf._peer.close()
        M, P = 64, 16
        pt = sig.firwin(M * P, 1.0 / M).astype(np.float32)
        nx = M * 4096
        lo, hi = mg.time_segments(nx, world, M, halo_len=(P - 1) * M)[rank]
        seg = torch.from_numpy(x[lo:hi]).cuda()
        st = mg.SegmentedFir(nb.PfbChannelizer(pt, M), rank, world, peer=True, halo_len=(P - 1) * M)
        rows = st.run(seg)
        torch.cuda.synchronize()
        allrows = gather_cpu(rows.contiguous())
        err = o.rel_rms(allrows.reshape(-1), o.pfb_channelizer(x[:nx], pt, M).reshape(-1))
        notes.append(("pfb", float(err)))
        ok &= bool(err < 1e-5)
        dist.barrier()
        st._peer.close()
        if rank == 0:
            q.put((ok, notes))
    finally:
        dist.destroy_process_group()


def test_time_segments_two_ranks_on_one_gpu_match_the_oracle():
    import torch
    import torch.multiprocessing as mp
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_one_gpu, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    ok, notes = q.get(timeout=5)
    assert ok is True, notes
