"""CPU tests of the host-side logic: metric reduction semantics against the reference goldens,
pair sharding, the world_size-2 gloo path of the metric all-reduce, and install() on the reference."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def sums_numpy(est, gt, maxdisp):
    """numpy restatement of what rag_loss_metrics_sums produces (test helper)."""
    out = np.zeros((est.shape[0], 8))
    for b in range(est.shape[0]):
        e, g = est[b].astype(np.float32), gt[b].astype(np.float32)
        pos = g > 0
        m = pos & (g < maxdisp)
        d = (e - g)[m]
        E = np.abs(g - e)[m]
        ad = np.abs(d)
        sl1 = np.where(ad < 1, np.float32(0.5) * d * d, ad - np.float32(0.5)).astype(np.float32)
        out[b] = [m.sum(), pos.sum(), sl1.astype(np.float64).sum(), E.astype(np.float64).sum(),
                  ((E > 3) & (E / np.abs(g[m]) > 0.05)).sum(), (E > 1).sum(), (E > 2).sum(), (E > 3).sum()]
    return out


def test_metrics_from_sums_matches_reference_golden():
    from rag_b200 import metrics as M

    z = np.load(os.path.join(GOLDEN, "metrics_b3_h12_w20.npz"))
    sums = torch.from_numpy(sums_numpy(z["est"], z["gt"], float(z["maxdisp"])))
    vec = M.metrics_from_sums(sums).numpy()
    for i, k in enumerate(M.KEYS):
        assert abs(vec[i] - float(z[k])) <= 2e-6 * max(1.0, abs(float(z[k]))), k


def test_shard_pairs_partitions_exactly():
    from rag_b200.dist import shard_pairs

    for n in (0, 1, 7, 8, 32, 33):
        for world in (1, 2, 3, 8):
            got = [i for r in range(world) for i in shard_pairs(n, r, world)]
            assert got == list(range(n))
            sizes = [len(shard_pairs(n, r, world)) for r in range(world)]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, batches, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from rag_b200 import dist as D
    from rag_b200 import metrics as M

    D.init("gloo")
    acc = M.MetricAccumulator("cpu")
    for i in D.shard_pairs(len(batches), rank, world):   # batches are sharded across ranks like pairs
        acc.update(torch.from_numpy(batches[i]))
    out = acc.mean()
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def test_metric_allreduce_gloo_world2():
    from rag_b200 import metrics as M

    rng = np.random.RandomState(0)
    batches = []
    for _ in range(5):
        gt = rng.rand(3, 10, 12).astype(np.float32) * 260 - 30
        est = gt + rng.randn(3, 10, 12).astype(np.float32) * 3
        batches.append(sums_numpy(est, gt, 192.0))
    single = M.MetricAccumulator("cpu")
    for s in batches:
        single.update(torch.from_numpy(s))
    want = single.mean(distributed=False)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, batches, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for k in M.KEYS:
        assert abs(got[k] - want[k]) <= 1e-12 * max(1.0, abs(want[k])), k


def _reference_modules():
    """(rag_model, mdenas_basicmodel, operations_3d): the unmodified reference's modules when oracle/_ref is installed,
    else stand-ins with the names install() rebinds (tests/_mirror_net.py)."""
    from oracle import refimport as R
    from tests._mirror_net import reference_modules

    if R.available():
        ref = R.import_reference()
        return ref.rag_model, ref.mdenas_basicmodel, ref.operations_3d
    return reference_modules()


def test_install_patches_the_reference_classes():
    """install() on the reference modules (the unmodified ones when installed, else stand-ins): the three forwards and the
    head classes are swapped, a network built afterwards is stateless in its head, and a CPU call fails loudly (no fallback)."""
    from rag_b200 import network as N
    from rag_b200.modules import Disp

    rm, mb, _ = _reference_modules()

    orig = rm.Network.forward
    done = N.install(rm, mb)
    try:
        assert rm.Network.forward is N.network_forward and rm.Network.search_forward is N.network_search_forward
        assert mb.BasicNetwork.forward is N.basic_network_forward and rm.Disp is Disp and mb.Disp is Disp
        assert set(done) == {"rag_model", "mdenas_basicmodel"}
        net = mb.BasicNetwork("cpu") if False else None  # constructing the supernet is slow; the class patch is what matters
        stub = type("S", (), {})()
        stub.maxdisp = 192
        stub.feature = lambda img, ta, p: torch.zeros(1, 12, 4, 8)
        stub.matching = lambda c, ta, p: c
        stub.disp = Disp(192)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            rm.Network.forward(stub, None, None, 0)
    finally:
        rm.Network.forward = orig


def test_install_uninstall_flags_and_upsample_proxy_on_the_reference():
    """install() / uninstall() bookkeeping on the reference modules (the unmodified ones when installed, else stand-ins; CPU:
    only the bindings, no kernels): every binding is restored, install(fuse_stem=False) after a fused install switches the
    default off, and install(upsample=True) exposes rag_b200.upsample.Upsample as rag_model.nn.Upsample while every other
    name still resolves to torch.nn."""
    from rag_b200 import network as N
    from rag_b200.upsample import Upsample

    rm, mb, ops3d = _reference_modules()

    N.uninstall()
    orig = (rm.Network.forward, rm.Network.search_forward, mb.BasicNetwork.forward, ops3d.ConvBR_3d.forward, rm.Disp, rm.nn)
    try:
        done = N.install(rm, mb, ops3d, fuse_stem=True, upsample=True)
        assert "nn.Upsample" in done["rag_model"] and done["operations_3d"] == ["ConvBR_3d.forward"]
        assert N._FUSE_STEM and N._STEM_AWARE
        assert rm.nn.Upsample is Upsample and rm.nn.Conv3d is torch.nn.Conv3d and rm.nn.ModuleList is torch.nn.ModuleList
        up = rm.nn.Upsample(size=[4, 6, 8], mode="trilinear", align_corners=True)       # what matching() builds per call
        x = torch.randn(1, 2, 2, 3, 4)
        assert torch.equal(up(x), torch.nn.Upsample(size=[4, 6, 8], mode="trilinear", align_corners=True)(x))   # CPU: nn.Upsample itself
        N.install(rm, mb)                                   # plain install afterwards: fusion default off again
        assert not N._FUSE_STEM
        stub = type("S", (), {"maxdisp": 48})()
        with pytest.raises(RuntimeError, match="no CPU fallback"):   # _volume() takes the materialising path -> CUDA-only kernel
            N._volume(stub, torch.zeros(1, 12, 2, 4), torch.zeros(1, 12, 2, 4), 48)
        stub.rag_b200_fuse_stem = True                       # per-instance opt-in while ConvBR_3d is fusion-aware
        from rag_b200.fused_stem import VirtualCostVolume

        assert isinstance(N._volume(stub, torch.zeros(1, 12, 2, 4), torch.zeros(1, 12, 2, 4), 48), VirtualCostVolume)
    finally:
        n = N.uninstall()
    assert n >= 8
    assert (rm.Network.forward, rm.Network.search_forward, mb.BasicNetwork.forward, ops3d.ConvBR_3d.forward, rm.Disp, rm.nn) == orig
    assert rm.nn is torch.nn and not N._FUSE_STEM and not N._STEM_AWARE


def test_refimport_installs_and_verifies_the_reference(tmp_path):
    """tools/install_ref.sh + oracle/refimport.py: the copy under oracle/_ref is byte-identical (sha256 manifest), imports, and the
    scoped CPU monkeypatch restores torch.cuda.current_device."""
    import subprocess

    from oracle import refimport as R

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = subprocess.run(["bash", os.path.join(root, "tools", "install_ref.sh")], capture_output=True, text=True)
    assert res.returncode in (0, 3), res.stderr               # 3: no checkout of the reference to install from
    if not R.available():
        pytest.skip("the unmodified reference is neither installed in oracle/_ref nor available to tools/install_ref.sh")
    assert R.verify_manifest() >= 20
    ref = R.import_reference(cpu_patch=True)
    g = R.make_genotype(ref, 0)
    assert g.normal.shape == (6, 2) and g.reduce.shape == (6, 2) and set(g.normal[:, 1]) <= {0, 1}
    before = torch.cuda.current_device
    with R.on_cpu():
        assert torch.cuda.current_device() == "cpu"
        d = ref.rag_model.Disp(24)(torch.randn(1, 1, 8, 2, 3))       # the unmodified reference head on CPU tensors
    assert torch.cuda.current_device is before and d.shape == (1, 6, 9)


def test_fp64_torch_evaluator_matches_the_numpy_evaluator():
    """oracle.disp_head_f64_torch (used on the GPU at BASELINE sizes) against oracle.disp_head_grad_f64 (numpy)."""
    from oracle import rag_oracle as O

    g = torch.Generator().manual_seed(3)
    for (b, dl, hl, wl, md) in [(2, 16, 5, 12, 48), (1, 20, 3, 4, 60), (1, 7, 2, 3, 24)]:
        cl = torch.randn(b, dl, hl, wl, generator=g)
        gd = torch.randn(b, 3 * hl, 3 * wl, generator=g)
        d, gg = O.disp_head_grad_f64(cl.numpy(), gd.numpy(), md)
        d2, g2 = O.disp_head_f64_torch(cl, md, gd)
        assert np.abs(d - d2.numpy()).max() <= 1e-12
        assert np.abs(gg - g2.numpy()).max() <= 1e-12 * max(1.0, np.abs(gg).max())
        d3, none = O.disp_head_f64_torch(cl, md)
        assert none is None and torch.equal(d3, d2)


def test_schedule_variant_ids_match_the_header():
    """rag_b200.pipeline's variant constants are the ones include/rag_b200.h defines, and every schedule names four of them."""
    import re

    from rag_b200 import pipeline as P_

    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "rag_b200.h")).read()
    macros = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define (RAG_[A-Z_]+) (\d+)\b", hdr)}
    for name in ("CV_FWD_SHARED", "CV_BWD_SHARED", "CV_FWD_SLIM", "CV_BWD_SLIM", "HEAD_FWD_SHARED", "HEAD_BWD_SHARED"):
        assert getattr(P_, name) == macros["RAG_" + name], name
    assert set(P_.SCHEDULES) >= {"coresident", "launch-order"}
    for vs in P_.SCHEDULES.values():
        assert len(vs) == 4 and all(v is None or isinstance(v, int) for v in vs)
    assert P_.SCHEDULES["coresident"] == (P_.CV_FWD_SLIM, P_.HEAD_FWD_SHARED, P_.CV_BWD_SLIM, P_.HEAD_BWD_SHARED)


def test_schedule_falls_back_to_default_kernels_outside_their_preconditions():
    """Widths that are not a multiple of four or a ratio other than 3 take the default entry points (variant None)."""
    from rag_b200.pipeline import OverlappedPath

    class _Shape:                                   # only .shape is read
        def __init__(self, *s):
            self.shape = s

    p = OverlappedPath.__new__(OverlappedPath)     # no CUDA streams on the CPU box
    p.maxdisp, p.variants = 192, (5, 4, 3, 3)
    assert p._variants(_Shape(1, 12, 8, 48), _Shape(1, 1, 64, 8, 48)) == (5, 4, 3, 3)
    assert p._variants(_Shape(1, 12, 8, 46), _Shape(1, 1, 64, 8, 46)) == (None, None, None, 3)
    assert p._variants(_Shape(1, 12, 8, 48), _Shape(1, 1, 48, 8, 48)) == (5, None, 3, None)
