"""Wide+deep from an HBM-resident set (sb_trainer_load_dataset_sparse): the resident entry points run sparse steps - the
dense block read in place by TMA, the index rows read through the step's batch descriptor, so that one captured graph
serves any batch - and they must compute what the dense net computes on the materialised one-hot matrix
(oracle.CleanTrainer / oracle.Bf16Trainer on wd.onehot_matrix), and what the host-fed sparse step computes."""
import ctypes
import importlib.util
import os
import socket

import numpy as np
import pytest

from oracle import shifu_oracle as so
from oracle import wide_deep as wd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SHAPES = {
    "small": dict(n_dense=21, vocab=[5, 9, 3, 17], hidden=[40, 24], acts=[so.ACT_TANH, so.ACT_RELU], B=130, lr=0.05),
    # BASELINE config 4: 500 dense + 5000 one-hot (50 categorical columns x 100 values), [1024, 512]
    "cfg4": dict(n_dense=500, vocab=[100] * 50, hidden=[1024, 512], acts=[so.ACT_RELU, so.ACT_RELU], B=1024, lr=0.01),
}
LEAD = 7          # rows in front of the first batch: every batch sits at a non-zero offset


def _problem(c, seed=3):
    """three batches of B rows at offsets LEAD, LEAD + B, LEAD + 2B; the last one ends at the last row of the set"""
    n_rows = LEAD + 3 * c["B"]
    Xd, idx, y, w = wd.synth_wide_deep_batch(n_rows, c["n_dense"], c["vocab"], seed)
    n_onehot = int(sum(c["vocab"]))
    net = so.NetDesc(c["n_dense"] + n_onehot, c["hidden"], c["acts"])
    return net, so.xavier_init(net, seed), (Xd, idx.astype(np.int32), y, w), n_onehot


def _trainer(sb, c, net, params, prec, n_onehot, opt=so.OPT_MOMENTUM, lr=None):
    desc = sb.make_desc(net.n_features, c["hidden"], c["acts"], optimizer=opt, learning_rate=c["lr"] if lr is None else lr,
                        max_batch=c["B"], precision=prec)
    t = sb.Trainer(desc)
    t.set_params(so.flatten_params(params))
    t.set_sparse(c["n_dense"], n_onehot, len(c["vocab"]))
    return t


def _oracle(net, params, prec, opt, lr, fused_out):
    cfg = so.OptConfig(kind=opt, lr=lr)
    return so.CleanTrainer(net, params, cfg) if prec != 1 else so.Bf16Trainer(net, params, cfg, fused_out=fused_out)


def _dense_batch(data, n_onehot, o, rows):
    Xd, idx, y, w = data
    X = np.concatenate([Xd[o:o + rows], wd.onehot_matrix(idx[o:o + rows], n_onehot)], axis=1)
    return X, y[o:o + rows], w[o:o + rows]


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 2, 1])
@pytest.mark.parametrize("shape", ["small", "cfg4"])
def test_resident_run_matches_oracle_and_host_fed_steps(sb, prec, shape):
    """10 steps through ONE run_resident call (tensor-core modes: two 4-step graphs + two single-step graphs), cycling
    through three batches at non-zero offsets, against the dense oracle on the one-hot matrix; in the fp32 modes also
    against the same steps through the host-fed sb_trainer_step_sparse"""
    c = SHAPES[shape]
    net, params, data, n_onehot = _problem(c)
    B, steps = c["B"], 10
    offs = [LEAD + (i % 3) * B for i in range(steps)]
    ref = _oracle(net, params, prec, so.OPT_MOMENTUM, c["lr"], c["hidden"][-1] <= 256)
    want = np.array([float(ref.step([_dense_batch(data, n_onehot, o, B)])[0]) for o in offs])
    with _trainer(sb, c, net, params, prec, n_onehot) as t:
        t.load_dataset_sparse(*data)
        t.run_resident(offs, B)
        got, theta = t.loss_history(1, steps), t.get_params()
    if prec == 1:       # the bounds of the resident bf16 curve in tests/test_benchmarked_paths.py
        assert np.abs(got - want).max() <= (1e-4 if shape == "cfg4" else 5e-4), (got, want)
        assert np.abs(theta - ref.theta).max() <= 5e-3
        return
    assert np.abs(got - want).max() <= 1e-4, (got, want)
    assert np.abs(theta - ref.theta).max() <= 1e-4
    Xd, idx, y, w = data
    with _trainer(sb, c, net, params, prec, n_onehot) as th:
        for o in offs:
            th.step_sparse(Xd[o:o + B], idx[o:o + B], y[o:o + B], w[o:o + B])
        theta_h = th.get_params()
    # not bit-equal: the order of the scatter's red.global.add is not fixed
    assert np.abs(theta - theta_h).max() <= 1e-5


@pytest.mark.gpu
def test_graph_replay_with_new_offsets_and_a_smaller_batch(sb):
    """the captured graphs serve any batch: two run_resident calls over different offsets, at rows < max_batch"""
    c = SHAPES["small"]
    net, params, data, n_onehot = _problem(c, seed=5)
    rows = c["B"] - 24
    runs = [[LEAD + k * 40 for k in (0, 1, 2, 3, 4, 5, 6, 7)], [LEAD + 3 * c["B"] - rows, 1, LEAD + 50, 0, 99, 3, 260, 11]]
    ref = _oracle(net, params, 2, so.OPT_MOMENTUM, c["lr"], True)
    with _trainer(sb, c, net, params, 2, n_onehot) as t:
        t.load_dataset_sparse(*data)
        for r, offs in enumerate(runs):
            want = np.array([float(ref.step([_dense_batch(data, n_onehot, o, rows)])[0]) for o in offs])
            t.run_resident(offs, rows)
            got = t.loss_history(1 + 8 * r, 8)
            assert np.abs(got - want).max() <= 1e-4, (r, got, want)
            assert np.abs(t.get_params() - ref.theta).max() <= 1e-4, r


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 2])
def test_accumulate_loss_and_profile_on_a_sparse_set(sb, prec):
    c = SHAPES["small"]
    net, params, data, n_onehot = _problem(c, seed=8)
    B = c["B"]
    offs = [LEAD, LEAD + B, LEAD + 2 * B]
    with _trainer(sb, c, net, params, prec, n_onehot, opt=so.OPT_SGD, lr=1.0) as t:
        t.load_dataset_sparse(*data)
        # loss only: no update
        L = so.loss_and_grads(net, params, *_dense_batch(data, n_onehot, offs[1], B))[0]
        assert abs(t.loss_resident(offs[1], B) - L) <= 1e-4
        # three accumulated mini-batch gradients, one update with their mean (plain SGD, lr = 1: theta moves by that mean)
        gsum = np.zeros(t.n_params, np.float32)
        for o in offs:
            loss = t.accumulate_resident(o, B)
            L, g, _ = so.loss_and_grads(net, params, *_dense_batch(data, n_onehot, o, B))
            assert abs(loss - L) <= 1e-4
            gsum += so.flatten_params(g)
        t.apply_accumulated(3)
        want = so.Optimizer(so.OptConfig(kind=so.OPT_SGD, lr=1.0), gsum.size).apply(so.flatten_params(params), gsum / np.float32(3))
        assert np.abs(t.get_grads() - gsum / np.float32(3)).max() <= 1e-4
        assert np.abs(t.get_params() - want).max() <= 1e-4
        names = [nm for nm, _ in t.profile_step(offs[2], B)]
    assert "embed_gather" in names and "embed_scatter" in names, names


@pytest.mark.gpu
def test_dense_and_sparse_sets_replace_each_other(sb):
    c = SHAPES["small"]
    net, params, data, n_onehot = _problem(c, seed=9)
    B = c["B"]
    offs = [LEAD + (i % 3) * B for i in range(5)]
    Xfull, y, w = _dense_batch(data, n_onehot, 0, len(data[0]))
    for order in (("sparse", "dense"), ("dense", "sparse")):
        ref = _oracle(net, params, 2, so.OPT_MOMENTUM, c["lr"], True)
        with _trainer(sb, c, net, params, 2, n_onehot) as t:
            for r, kind in enumerate(order):
                if kind == "sparse":
                    t.load_dataset_sparse(*data)
                else:
                    t.load_dataset(Xfull, y, w)
                want = np.array([float(ref.step([_dense_batch(data, n_onehot, o, B)])[0]) for o in offs])
                t.run_resident(offs, B)
                assert np.abs(t.loss_history(1 + 5 * r, 5) - want).max() <= 1e-4, (order, kind)
                assert np.abs(t.get_params() - ref.theta).max() <= 1e-4, (order, kind)


@pytest.mark.gpu
def test_load_argument_checks(sb):
    torch = pytest.importorskip("torch")
    c = SHAPES["small"]
    net, params, (Xd, idx, y, w), n_onehot = _problem(c)
    desc = sb.make_desc(net.n_features, c["hidden"], c["acts"], max_batch=c["B"], precision=1)
    with sb.Trainer(desc) as t:
        with pytest.raises(sb.ShifuB200Error) as e:
            t.load_dataset_sparse(Xd, idx, y, w)
        assert e.value.code == sb.capi.SB_ERR_STATE
        t.set_sparse(c["n_dense"], n_onehot, len(c["vocab"]))
        t.load_dataset_sparse(Xd, idx, y, w)
        for bad_value in (n_onehot, -2):
            bad = idx.copy()
            bad[len(bad) - 1, 2] = bad_value
            with pytest.raises(sb.ShifuB200Error) as e:
                t.load_dataset_sparse(Xd, bad, y, w)                     # host array
            assert e.value.code == sb.capi.SB_ERR_INVALID
            dev = torch.from_numpy(bad).to("cuda:0")
            torch.cuda.synchronize()
            da = sb.capi.DeviceArray(ctypes.cast(ctypes.c_void_p(dev.data_ptr()), sb.capi._f32p), bad.shape, owner=False)
            with pytest.raises(sb.ShifuB200Error) as e:
                t.load_dataset_sparse(Xd, da, y, w)                      # device array
            assert e.value.code == sb.capi.SB_ERR_INVALID
        # the rejected loads left the set that was loaded before
        assert t.loss_resident(LEAD, c["B"]) > 0
        with pytest.raises(sb.ShifuB200Error) as e:
            t.set_sparse(c["n_dense"] - 1, n_onehot + 1, len(c["vocab"]))   # another shape while a sparse set is loaded
        assert e.value.code == sb.capi.SB_ERR_STATE


def _replica_problem():
    c = dict(n_dense=64, vocab=[20, 30, 14], hidden=[96, 48], acts=[so.ACT_RELU, so.ACT_TANH], B=256)
    n_onehot = int(sum(c["vocab"]))
    net = so.NetDesc(c["n_dense"] + n_onehot, c["hidden"], c["acts"])
    return c, n_onehot, net


@pytest.mark.gpu
@pytest.mark.parametrize("prec", [0, 1])
def test_two_replicas_on_one_gpu_match_the_data_parallel_oracle(sb, monkeypatch, prec):
    """W = 2 in-process replicas over the peer exchange kernels (fp32: flag-and-pull, bf16: LL): the layer-0 gradient of a
    sparse step is exchanged behind everything, also inside the multi-step graphs"""
    monkeypatch.setenv("SB_XCHG_BLOCKS", "8")
    monkeypatch.setenv("SB_XCHG_TIMEOUT_S", "60")
    c, n_onehot, net = _replica_problem()
    W, B, n_steps = 2, c["B"], 10
    kind, lr = (so.OPT_ADAM, 0.003) if prec == 0 else (so.OPT_MOMENTUM, 0.05)
    params = so.xavier_init(net, 4)
    shards = [wd.synth_wide_deep_batch(3 * B, c["n_dense"], c["vocab"], 40 + 17 * r) for r in range(W)]
    desc = sb.make_desc(net.n_features, c["hidden"], c["acts"], optimizer=kind, learning_rate=lr, max_batch=B, precision=prec)
    ts = [sb.Trainer(desc, device=0, nccl_id=None, rank=r, world=W) for r in range(W)]
    for t in ts:
        t.set_peer_pointers([x.exchange_base for x in ts])
        t.set_params(so.flatten_params(params))
        t.set_sparse(c["n_dense"], n_onehot, len(c["vocab"]))
    for t, (Xd, idx, y, w) in zip(ts, shards):
        t.load_dataset_sparse(Xd, idx, y, w)
    for s0 in range(0, n_steps, 4):
        offs = [((s0 + k) % 3) * B for k in range(min(4, n_steps - s0))]
        for t in ts:
            t.run_resident(offs, B)
    for t in ts:
        t.sync()
    ref = _oracle(net, params, prec, kind, lr, True)
    want = np.array([ref.step([_dense_batch(sh, n_onehot, (s % 3) * B, B) for sh in shards]) for s in range(n_steps)], np.float64)
    got = np.stack([t.loss_history(1, n_steps) for t in ts], axis=1)
    thetas = [t.get_params() for t in ts]
    grads = [t.get_grads() for t in ts]
    preds = [t.predict_sparse(shards[0][0][:300], shards[0][1][:300]) for t in ts]
    for t in ts:
        t.close()
    np.testing.assert_array_equal(thetas[0], thetas[1])
    np.testing.assert_array_equal(grads[0], grads[1])
    np.testing.assert_array_equal(preds[0], preds[1])
    tol_l, tol_p = (1e-4, 1e-4) if prec == 0 else (1e-3, 5e-3)
    assert np.abs(got - want).max() <= tol_l, (got, want)
    if kind == so.OPT_ADAM:      # see tests/test_benchmarked_paths.py: Adam moves noise-level coordinates by +-lr
        assert np.linalg.norm(thetas[0] - ref.theta) / np.linalg.norm(ref.theta) <= 1e-2
    else:
        assert np.abs(thetas[0] - ref.theta).max() <= tol_p


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _two_gpu_rank_main(rank, world, port, out_dir, precision):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    import shifu_tensorflow_b200 as sb
    from shifu_tensorflow_b200 import dist_util as du
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("SB_XCHG_TIMEOUT_S", "60")
    dist.init_process_group("gloo", rank=rank, world_size=world)
    c, n_onehot, net = _replica_problem()
    desc = sb.make_desc(net.n_features, c["hidden"], c["acts"], optimizer=so.OPT_MOMENTUM, learning_rate=0.05, max_batch=c["B"],
                        precision=precision)
    t = sb.Trainer(desc, device=rank, nccl_id=None, rank=rank, world=world)
    du.enable_peer_exchange(dist, t, world)
    t.set_params(so.flatten_params(so.xavier_init(net, 4)))
    t.set_sparse(c["n_dense"], n_onehot, len(c["vocab"]))
    t.load_dataset_sparse(*wd.synth_wide_deep_batch(3 * c["B"], c["n_dense"], c["vocab"], 40 + 17 * rank))
    t.run_resident([(s % 3) * c["B"] for s in range(10)], c["B"])
    hist = t.loss_history(1, 10)
    theta, grads = t.get_params(), t.get_grads()
    dist.barrier()
    np.savez(os.path.join(out_dir, "r%d.npz" % rank), theta=theta, grads=grads, losses=np.array(hist))
    t.close()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [1, 2])
def test_two_gpu_sparse_resident_run_matches_oracle(sb, tmp_path, precision):
    """the same on two real GPUs over CUDA-IPC peer memory, the schedule of a multi-GPU run"""
    if sb.capi.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_two_gpu_rank_main, args=(world, _free_port(), str(tmp_path), precision), nprocs=world, join=True)
    r = [np.load(str(tmp_path / ("r%d.npz" % i))) for i in range(world)]
    np.testing.assert_array_equal(r[0]["theta"], r[1]["theta"])
    np.testing.assert_array_equal(r[0]["grads"], r[1]["grads"])
    c, n_onehot, net = _replica_problem()
    shards = [wd.synth_wide_deep_batch(3 * c["B"], c["n_dense"], c["vocab"], 40 + 17 * k) for k in range(world)]
    ref = _oracle(net, so.xavier_init(net, 4), precision, so.OPT_MOMENTUM, 0.05, True)
    want = np.array([ref.step([_dense_batch(sh, n_onehot, (s % 3) * c["B"], c["B"]) for sh in shards]) for s in range(10)])
    tol_l, tol_p = (1e-4, 1e-4) if precision == 2 else (1e-3, 5e-3)
    for k in range(world):
        assert np.abs(r[k]["losses"] - want[:, k]).max() <= tol_l
    assert np.abs(r[0]["theta"] - ref.theta).max() <= tol_p


def test_bench_wide_deep_counts_config4():
    """scripts/bench_wide_deep.py's FLOP / byte counts of config 4 (500 dense + 50 x 100 one-hot, [1024, 512])"""
    spec = importlib.util.spec_from_file_location("bench_wide_deep", os.path.join(ROOT, "scripts", "bench_wide_deep.py"))
    bw = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bw)
    cnt = bw.work_per_row(500, [100] * 50, [1024, 512])
    assert cnt["sparse"]["gemm_flop"] == 5_196_800
    assert cnt["dense_onehot"]["gemm_flop"] == 25_676_800
    assert cnt["sparse"]["embed_adds"] == 2 * 50 * 1024
    assert cnt["sparse"]["bytes"] == 1008 + 200 + 8
    assert cnt["dense_onehot"]["bytes"] == 11_008 + 8
