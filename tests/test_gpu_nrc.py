"""GPU parity: the NRC network (fused hash-grid/one-blob/identity encoding + tcgen05 MLP inference and training step;
the CUDA-core training kernel for networks of more than 3 hidden layers) vs the CPU oracle.  Tensor-core accumulation order is hardware-defined, so the bar is
<= 1e-3 relative L2 on inference (BASELINE.json north_star) and agreement of loss curves / weights on training."""
import numpy as np
import pytest

from gfxexp_b200 import engine

pytestmark = pytest.mark.gpu


def _queries(n, seed=0):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.0, 1.0, size=(n, 14)).astype(np.float32)


def _rel_l2(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-20))


@pytest.mark.parametrize("hidden,amp", [(2, 1e-4), (2, 0.5), (5, 0.5)])
def test_inference_matches_oracle(gfx_ctx, oracle, hidden, amp):
    import torch
    onet = oracle.OracleNrc(hidden, 1e-2)
    params = engine.random_nrc_params(onet.num_params, onet.num_matrix_weights, seed=7 + hidden, grid_amplitude=amp)
    onet.set_params(params)
    gnet = engine.NeuralRadianceCache(gfx_ctx, hidden, 1e-2)
    assert gnet.num_params == onet.num_params
    gnet.set_params(params)
    n = 128 * 300
    q = _queries(n, 5)
    q[:64, :3] = 0.0      # grid corners / cell boundaries
    q[64:128, :3] = 1.0
    dq = torch.from_numpy(q).cuda()
    out = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    gnet.infer(dq, out, n)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    want = onet.infer(q)
    assert np.isfinite(got).all()
    assert _rel_l2(got, want) <= 1e-3, _rel_l2(got, want)
    gnet.close()


def test_split_encoding_is_bit_exact(gfx_ctx, oracle):
    """the encoded network input of the split inference path (positions packed, one hash-grid level per CTA with the level's
    table staged in shared memory by TMA, one-blob + identity in the MLP kernel) equals the oracle's - which is pinned bit for
    bit against tiny-cuda-nn's kernel_grid / kernel_one_blob_soa (tests/test_gpu_tcnn_ref.py) - in every half"""
    import torch
    onet = oracle.OracleNrc(2, 1e-2)
    params = engine.random_nrc_params(onet.num_params, onet.num_matrix_weights, seed=3, grid_amplitude=0.5)
    onet.set_params(params)
    gnet = engine.NeuralRadianceCache(gfx_ctx, 2, 1e-2)
    gnet.set_params(params)
    n = 128 * 150 + 128  # not a multiple of the replica count
    q = _queries(n, 9)
    rng = np.random.default_rng(4)
    q[:64, :3] = 0.0
    q[64:128, :3] = 1.0
    q[128:256, :3] = (rng.integers(0, 17, size=(128, 3)) / 16.0).astype(np.float32)   # level-0 cell corners
    q[256:384, :3] = (rng.integers(0, 513, size=(128, 3)) / 512.0).astype(np.float32)  # finer cell corners
    q[384:512, 3:8] = rng.choice([0.0, 0.25, 0.5, 0.75, 1.0], size=(128, 5)).astype(np.float32)
    got = gnet.encode(torch.from_numpy(q).cuda(), n).view(np.uint16)
    want = onet.encode(q).view(np.uint16).reshape(n, 64)
    bad = np.argwhere(got != want)
    assert bad.size == 0, f"{len(bad)} halves differ, first {bad[:5].tolist()}"
    gnet.close()


def test_fused_and_split_inference_agree(gfx_ctx):
    """Queries or predictions that are not 16-byte aligned (here: views 4 bytes into their buffers) take the fused kernel
    (hash-grid gathers from L2 inside the MLP kernel); aligned ones take the split path.  Both feed the same halves to the
    same tcgen05 MLP: identical radiance"""
    import torch
    gnet = engine.NeuralRadianceCache(gfx_ctx, 2, 1e-2)
    gnet.set_params(engine.random_nrc_params(gnet.num_params, 64 * 64 * 2 + 16 * 64, seed=5, grid_amplitude=0.5))
    n = 128 * 77
    dq = torch.from_numpy(_queries(n, 2)).cuda()
    dq_offset = torch.empty(n * 14 + 1, device="cuda")[1:].view(n, 14)
    dq_offset.copy_(dq)
    split = torch.empty((n, 3), device="cuda")
    fused_in = torch.empty((n, 3), device="cuda")
    fused_out = torch.empty(n * 3 + 1, device="cuda")[1:].view(n, 3)
    assert dq.data_ptr() % 16 == 0 and split.data_ptr() % 16 == 0 and fused_in.data_ptr() % 16 == 0
    assert dq_offset.data_ptr() % 16 == 4 and fused_out.data_ptr() % 16 == 4
    gnet.infer(dq, split, n)
    gnet.infer(dq_offset, fused_in, n)
    gnet.infer(dq, fused_out, n)
    torch.cuda.synchronize()
    assert torch.equal(split, fused_in)
    assert torch.equal(split, fused_out)
    gnet.close()


def test_infer_rejects_unpadded_batch(gfx_ctx):
    import torch
    gnet = engine.NeuralRadianceCache(gfx_ctx, 2, 1e-2)
    dq = torch.zeros((100, 14), device="cuda")
    out = torch.zeros((100, 3), device="cuda")
    with pytest.raises(engine.GfxError):
        gnet.infer(dq, out, 100)  # network_interface.cu:143 requires numData % 128 == 0
    gnet.close()


def _train_against_oracle(gfx_ctx, oracle, hidden):
    import torch
    onet = oracle.OracleNrc(hidden, 1e-2)
    params = engine.random_nrc_params(onet.num_params, onet.num_matrix_weights, seed=11)
    onet.set_params(params)
    gnet = engine.NeuralRadianceCache(gfx_ctx, hidden, 1e-2)
    gnet.set_params(params)
    n = 4096
    q = _queries(n, 9)
    target = np.stack([0.5 + 0.4 * np.sin(6 * q[:, 0]), q[:, 1] * q[:, 8], 0.3 + 0.5 * q[:, 2]], axis=1).astype(np.float32)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(target).cuda()
    gl, ol = [], []
    for _ in range(12):
        gl.append(gnet.train(dq, dt, n, want_loss=True))
        ol.append(onet.train(q, target))
    gl, ol = np.array(gl), np.array(ol)
    assert np.isfinite(gl).all()
    assert np.abs(gl - ol).max() <= 0.05 * ol.max(), (gl, ol)
    assert gl[-1] < 0.5 * gl[0]
    # inference after training (EMA weights) agrees
    out = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    gnet.infer(dq, out, n)
    torch.cuda.synchronize()
    assert _rel_l2(out.cpu().numpy(), onet.infer(q)) <= 2e-2
    gnet.close()


def test_training_tracks_oracle(gfx_ctx, oracle):
    """2 hidden layers: the tcgen05 training kernel (forward, data and weight gradients as MMAs)"""
    _train_against_oracle(gfx_ctx, oracle, 2)


def test_cuda_core_training_tracks_oracle(gfx_ctx, oracle):
    """4 hidden layers, the shallowest network whose activation tiles do not fit the tcgen05 training kernel's shared
    memory: the CUDA-core training kernel"""
    _train_against_oracle(gfx_ctx, oracle, 4)


def test_tensor_core_training_is_deterministic(gfx_ctx):
    import torch
    n = 4096
    q = _queries(n, 22)
    target = np.stack([q[:, 0], q[:, 1], q[:, 2]], axis=1).astype(np.float32)
    dq, dt = torch.from_numpy(q).cuda(), torch.from_numpy(target).cuda()
    outs = []
    for _ in range(2):
        net = engine.NeuralRadianceCache(gfx_ctx, 2, 1e-2)
        net.set_params(engine.random_nrc_params(net.num_params, 64 * 64 * 2 + 16 * 64, seed=5))
        for _ in range(6):
            net.train(dq, dt, n)
        out = torch.empty((n, 3), dtype=torch.float32, device="cuda")
        net.infer(dq, out, n)
        torch.cuda.synchronize()
        outs.append(out.cpu().numpy())
        net.close()
    assert np.array_equal(outs[0], outs[1])
