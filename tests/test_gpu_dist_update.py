"""-m gpu, needs >= 2 GPUs (skips on a machine with one): the row-block partitioned large-map update
(BASELINE config 4).  Two ranks hold replicas of the same filter, each updates only its rows of
Sigma, NCCL carries the W / V panels and the row blocks; every rank must end with the same state as
a single-GPU filter and as the CPU oracle."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, out_dir, n_features, n_frames, lookahead_min_n):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")]
    import torch
    import torch.distributed as dist
    import ekfb200
    pkg = ekfb200.load_package()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    if lookahead_min_n:   # force the pipelined (look-ahead) partitioned update, normally used from n = 6000
        os.environ["EKF_LOOKAHEAD_MIN_N"] = str(lookahead_min_n)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    sc = pkg.synth.Scene(n_features=n_features, n_frames=n_frames, seed=55)
    cfg = pkg.default_config(**sc.config_overrides())
    f = pkg.VSlamFilter(cfg, feature_capacity=n_features + 4, device=rank)
    f.captureNewFrame(sc.frame(0), sc.stamps[0])
    for p in sc.feature_pixels:
        f.addFeature(*p)
    pkg.dist.attach_row_partition(f, dist, torch.device("cuda", rank))
    stats = []
    for t in range(1, n_frames):
        f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, n_features))
        s = f.stats(); stats.append((s.n_matched, s.n_li, s.n_hi))
    mu, S = f.get_full()
    info = f.dist_info()
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), mu=mu, S=S, stats=np.array(stats), bytes=info["allgather_bytes"], world=info["world"], peer=int(info["peer_memory"]))
    f.dist_detach()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("n_features,lookahead_min_n", [(40, 0), (150, 0), (150, 100), (330, 100)])
def test_row_partitioned_update_matches_single_gpu_and_oracle(gpu_pkg, orc, tmp_path, n_features, lookahead_min_n):
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from helpers import TOL, make_pair, relerr, seed_features
    world, n_frames = 2, 4
    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path), n_features, n_frames, lookahead_min_n), nprocs=world, join=True)
    r = [np.load(tmp_path / f"r{k}.npz") for k in range(world)]
    assert int(r[0]["world"]) == 2 and int(r[0]["bytes"]) > 0
    # the panels travel by peer-memory stores unless EKF_DIST_P2P=0 (then by NCCL collectives)
    assert int(r[0]["peer"]) == (0 if os.environ.get("EKF_DIST_P2P") == "0" else 1)
    # replicas stay identical across ranks (same arithmetic on the same data)
    assert np.array_equal(r[0]["mu"], r[1]["mu"]) and np.array_equal(r[0]["S"], r[1]["S"])
    sc = gpu_pkg.synth.Scene(n_features=n_features, n_frames=n_frames, seed=55)
    g, o = make_pair(gpu_pkg, orc, sc)
    g.set_symmetric_downdate(False)
    seed_features(g, sc); seed_features(o, sc)
    for t in range(1, n_frames):
        for f in (g, o):
            f.captureNewFrame(sc.frame(t), sc.stamps[t]); f.predict(); f.update(sc.picks(t, n_features))
    mg, Sg = g.get_full(); mo, So = o.get_full()
    assert r[0]["mu"].shape == mg.shape
    tol_sg = 1e-10 if lookahead_min_n else 1e-12   # the look-ahead correction reorders two subtractions per element
    assert relerr(r[0]["mu"], mg) <= tol_sg and relerr(r[0]["S"], Sg) <= tol_sg, "partitioned vs single-GPU (full-square downdate)"
    assert relerr(r[0]["mu"], mo) <= 1e-8 and relerr(r[0]["S"], So) <= 1e-8, "partitioned vs oracle (free running)"
    print(f"N={n_features}: partitioned vs single GPU mu {relerr(r[0]['mu'], mg):.1e} Sigma {relerr(r[0]['S'], Sg):.1e}; "
          f"vs oracle mu {relerr(r[0]['mu'], mo):.1e} Sigma {relerr(r[0]['S'], So):.1e}; all-gather bytes/rank {int(r[0]['bytes'])}")
