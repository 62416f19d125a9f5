"""CPU: sharding a fan-out call (A audio clips x K sequences each) by audio clip, over gloo (no kernels involved)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def test_fanout_shard_range():
    from fdm_b200.parallel import fanout_shard_range
    n_audio, k = 8, 3
    for world in (1, 2, 4):
        per = n_audio // world
        got = [fanout_shard_range(n_audio, k, r, world) for r in range(world)]
        assert got == [((r * per, per), (r * per * k, per * k)) for r in range(world)]
        # the ranks' sequence ranges tile 0 .. n_audio*k in order, and each clip's k sequences stay on its rank
        seqs = [s for _, (s0, n) in got for s in range(s0, s0 + n)]
        assert seqs == list(range(n_audio * k))
        for (a0, na), (s0, n) in got:
            assert {s // k for s in range(s0, s0 + n)} == set(range(a0, a0 + na))
    assert fanout_shard_range(5, 7, 0, 1) == ((0, 5), (0, 35))
    with pytest.raises(ValueError):
        fanout_shard_range(6, 2, 0, 4)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, n_audio, k, q):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path[:0] = [root, os.path.join(root, "face-diffusion-model_b200")]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from fdm_b200.parallel import fanout_shard_range, gather_clips
    from oracle.philox_ref import philox_normal
    (a0, na), (clip_index0, n) = fanout_shard_range(n_audio, k, rank, world)
    audio = torch.arange(a0, a0 + na, dtype=torch.float32)  # this rank's audio clips only
    # stand-in for the per-rank fan-out job: sequence i uses audio clip i // k, noise keyed by the global sequence index
    local = torch.stack([torch.from_numpy(philox_normal(7, clip_index0 + i, 3, 64)).view(4, 16) + 1000 * audio[i // k]
                         for i in range(n)])
    q.put((rank, gather_clips(local).numpy()))
    dist.barrier()
    dist.destroy_process_group()


def test_fanout_sharded_sampling_is_world_size_invariant():
    from oracle.philox_ref import philox_normal
    n_audio, k, world = 4, 3, 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_audio, k, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # the unsharded call: audio.repeat_interleave(k, 0) order, noise of sequence s keyed by s
    ref = np.stack([philox_normal(7, s, 3, 64).reshape(4, 16) + 1000 * (s // k) for s in range(n_audio * k)])
    for r in range(world):
        assert got[r].shape == (n_audio * k, 4, 16)
        assert np.array_equal(got[r], ref)
