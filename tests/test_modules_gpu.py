"""Module-level GPU tests: the reference's dense-equivalence test (test/test_conv.py:247-357)
run through SparseConv3d / SubMConv3d with autograd, against torch conv3d on the densified input
(tests.util.dense_conv_case and live); indice_key caching; inverse conv; AMP."""
import numpy as np
import pytest
import torch

from tests.util import dense_conv_case, random_cloud, rel_l2

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("algo_name", ["Native", "MaskImplicitGemm"])
@pytest.mark.parametrize("tag,k,s,p,d", [("k3s2p1d1", 3, 2, 1, 1), ("k3s1p1d1", 3, 1, 1, 1),
                                         ("k2s2p0d1", 2, 2, 0, 1)])
def test_sparse_conv3d_equals_dense_golden(tag, k, s, p, d, algo_name, cuda_dev):
    import spconv_b200.pytorch as spconv
    from spconv_b200.core import ConvAlgo
    g = dense_conv_case()
    inds, feats, shape = g["inds"], g["feats"], [int(v) for v in g["shape"]]
    w, y, dy = g[f"{tag}_w"], g[f"{tag}_y"], g[f"{tag}_dy"]
    C, K = feats.shape[1], w.shape[0]
    layer = spconv.SparseConv3d(C, K, k, s, p, d, bias=False, algo=ConvAlgo[algo_name]).to(cuda_dev)
    with torch.no_grad():
        layer.weight.copy_(torch.from_numpy(w))
    x_feats = torch.from_numpy(feats).to(cuda_dev).requires_grad_(True)
    x = spconv.SparseConvTensor(x_feats, torch.from_numpy(inds).to(cuda_dev), shape, 2)
    out = layer(x)
    dense = out.dense()
    assert tuple(dense.shape) == y.shape
    assert np.abs(dense.detach().cpu().numpy() - y).max() < 1e-4            # test_conv.py:330
    dense.backward(torch.from_numpy(dy).to(cuda_dev))
    # the expected gradients come from torch dense conv3d with dy masked to the active outputs
    # (tests.util.dense_conv_case); the sparse op defines gradients through those only
    ref_dw, ref_dx = g[f"{tag}_dw"], g[f"{tag}_dx"]
    assert np.abs(layer.weight.grad.cpu().numpy() - ref_dw).max() < 1e-3
    assert np.abs(x_feats.grad.cpu().numpy() - ref_dx).max() < 1e-4


@pytest.mark.parametrize("algo_name", ["Native", "MaskImplicitGemm"])
def test_subm_equals_dense_on_active_set(algo_name, cuda_dev):
    import spconv_b200.pytorch as spconv
    from spconv_b200.core import ConvAlgo
    rng = np.random.default_rng(484)
    shape = [19, 18, 17]
    feats, inds = random_cloud(rng, shape, [1500, 1500], 32)
    layer = spconv.SubMConv3d(32, 48, 3, dilation=2, bias=True, algo=ConvAlgo[algo_name]).to(cuda_dev)
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev), torch.from_numpy(inds).to(cuda_dev), shape, 2)
    out = layer(x)
    assert out.indices is x.indices and out.spatial_shape == shape
    dense_in = x.dense().cpu()
    w = layer.weight.detach().cpu().permute(0, 4, 1, 2, 3).contiguous()
    ref = torch.nn.functional.conv3d(dense_in, w, layer.bias.detach().cpu(), padding=2, dilation=2)
    ref_rows = ref[inds[:, 0], :, inds[:, 1], inds[:, 2], inds[:, 3]]
    assert (out.features.cpu() - ref_rows).abs().max() < 1e-4


def test_indice_key_reuse_and_errors(cuda_dev):
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch import ops
    rng = np.random.default_rng(1)
    shape = [24, 24, 24]
    feats, inds = random_cloud(rng, shape, [2500], 16)
    net = spconv.SparseSequential(
        spconv.SubMConv3d(16, 16, 3, indice_key="subm1"), torch.nn.ReLU(),
        spconv.SubMConv3d(16, 16, 3, indice_key="subm1"), torch.nn.ReLU(),
        spconv.SparseConv3d(16, 32, 3, 2, 1, indice_key="down1"),
        spconv.SubMConv3d(32, 32, 3, indice_key="subm2"),
        spconv.SparseInverseConv3d(32, 16, 3, indice_key="down1"),
    ).to(cuda_dev).half()
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev).half(), torch.from_numpy(inds).to(cuda_dev), shape, 1)
    ops.launch_count(reset=True)
    y = net(x)
    assert set(y.indice_dict) == {"subm1", "down1", "subm2"}
    # the second subm1 layer reuses the cached rulebook; the inverse conv restores the input set
    assert y.indices.shape == x.indices.shape and torch.equal(y.indices, x.indices)
    assert y.spatial_shape == shape and y.features.shape == (2500, 16)
    assert torch.isfinite(y.features.float()).all()
    # same key, different kernel size -> reference error text
    bad = spconv.SubMConv3d(16, 16, 5, indice_key="subm1", large_kernel_fast_algo=True).to(cuda_dev).half()
    with pytest.raises(ValueError, match="same kernel size"):
        bad(net[0](x))
    # a regular conv cannot reuse a key
    dup = spconv.SparseConv3d(32, 16, 3, 2, 1, indice_key="down1").to(cuda_dev).half()
    with pytest.raises(AssertionError, match="only support reuse subm indices"):
        dup(net[4](net[0](x)))
    # different algo on a shared key
    from spconv_b200.core import ConvAlgo
    nat = spconv.SubMConv3d(16, 16, 3, indice_key="subm1", algo=ConvAlgo.Native).to(cuda_dev).half()
    with pytest.raises(AssertionError, match="same algo"):
        nat(net[0](x))


def test_inverse_conv_matches_oracle(oracle, cuda_dev):
    import spconv_b200.pytorch as spconv
    rng = np.random.default_rng(2)
    shape = [20, 20, 20]
    feats, inds = random_cloud(rng, shape, [1800], 16)
    down = spconv.SparseConv3d(16, 32, 3, 2, 1, bias=False, indice_key="d").to(cuda_dev)
    up = spconv.SparseInverseConv3d(32, 16, 3, indice_key="d", bias=False).to(cuda_dev)
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev), torch.from_numpy(inds).to(cuda_dev), shape, 1)
    mid = down(x)
    y = up(mid)
    o, p, n = oracle.get_indice_pairs(inds, 1, shape, [3] * 3, [2] * 3, [1] * 3, [1] * 3, [0] * 3, False)
    r_mid = oracle.indice_conv(feats, down.weight.detach().cpu().numpy(), p, n, o.shape[0], False, False)
    r_y = oracle.indice_conv(r_mid, up.weight.detach().cpu().numpy(), p, n, feats.shape[0], True, False)
    assert np.abs(mid.features.detach().cpu().numpy() - r_mid).max() < 1e-4
    assert np.abs(y.features.detach().cpu().numpy() - r_y).max() < 1e-3


def test_training_step_matches_fp32_oracle_and_amp(oracle, cuda_dev):
    import spconv_b200.pytorch as spconv
    rng = np.random.default_rng(3)
    shape = [24, 24, 24]
    feats, inds = random_cloud(rng, shape, [3000], 32)
    layer = spconv.SubMConv3d(32, 64, 3, bias=True).to(cuda_dev)
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev), torch.from_numpy(inds).to(cuda_dev), shape, 1)
    layer.train()
    with torch.autocast("cuda", dtype=torch.float16):
        y = layer(x)                       # custom_fwd casts features and weight to fp16
    assert y.features.dtype == torch.float16
    loss = y.features.float().square().mean()
    loss.backward()
    _, p, n = oracle.get_indice_pairs(inds, 1, shape, [3] * 3, [1] * 3, [1] * 3, [1] * 3, [0] * 3, True)
    w = layer.weight.detach().half().float().cpu().numpy()
    f16 = torch.from_numpy(feats).half().float().numpy()
    ref = oracle.indice_conv(f16, w, p, n, 3000, False, True) + layer.bias.detach().cpu().numpy()
    assert rel_l2(y.features.float().detach().cpu().numpy(), ref) < 1e-2
    assert layer.weight.grad is not None and layer.weight.grad.dtype == torch.float32
    assert layer.bias.grad is not None
    dout = (2.0 / ref.size) * ref
    _, ref_dw = oracle.indice_conv_backward(f16, w, dout, p, n, False, True)
    assert rel_l2(layer.weight.grad.cpu().numpy(), ref_dw) < 3e-2


def test_fused_bn_act_block_equals_unfused(cuda_dev):
    """north_star "fused BN/act": conv -> BatchNorm1d -> ReLU folded into ONE kernel launch per layer
    (weights + bias folded on the host, bias + activation in the GEMM epilogue); reference recipe
    example/fuse_bn_act.py:36-86"""
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch import ops
    rng = np.random.default_rng(4)
    shape = [20, 20, 20]
    feats, inds = random_cloud(rng, shape, [2500], 32)
    net = spconv.SparseSequential(
        spconv.SubMConv3d(32, 32, 3, bias=False, indice_key="a"), torch.nn.BatchNorm1d(32), torch.nn.ReLU(),
        spconv.SparseConv3d(32, 64, 3, 2, 1, bias=True), torch.nn.BatchNorm1d(64), torch.nn.LeakyReLU(0.1),
        spconv.SubMConv3d(64, 64, 3, bias=False, indice_key="b"), torch.nn.BatchNorm1d(64),
    ).to(cuda_dev)
    with torch.no_grad():
        for m in net:
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.uniform_(-0.5, 0.5)
                m.running_var.uniform_(0.5, 2.0)
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.5, 0.5)
    net.eval()
    fused = spconv.fuse_bn_act_sequential(net)
    assert len(fused) == 3 and all(isinstance(m, spconv.SparseConvolution) for m in fused)
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev), torch.from_numpy(inds).to(cuda_dev), shape, 1)
    with torch.no_grad():
        ref = net(x)
        ops.launch_count(reset=True)
        got = fused(x)
    assert torch.equal(ref.indices, got.indices)
    assert (ref.features - got.features).abs().max() < 1e-4 * max(1.0, float(ref.features.abs().max()))


@pytest.mark.parametrize("subm", [True, False])
def test_mask_split_implicit_gemm_is_a_real_split(subm, oracle, cuda_dev):
    """ConvAlgo.MaskSplitImplicitGemm (spconv/pytorch/ops.py:494-503): two mask splits (low / high
    offsets), each sorted on its own, one kernel pass per split; results equal the unsplit algo."""
    import spconv_b200.pytorch as spconv
    from spconv_b200.core import ConvAlgo
    from spconv_b200.pytorch import ops
    rng = np.random.default_rng(21)
    shape = [20, 22, 18]
    feats, inds = random_cloud(rng, shape, [2600], 32)
    d_inds = torch.from_numpy(inds).to(cuda_dev)
    k, s, p = ([3] * 3, [1] * 3, [1] * 3) if subm else ([3] * 3, [2] * 3, [1] * 3)
    res = ops.get_indice_pairs_implicit_gemm(d_inds, 1, shape, ConvAlgo.MaskSplitImplicitGemm, k, s, p, [1] * 3,
                                             [0] * 3, subm, False, is_train=True)
    out_inds, _, pair_fwd, pair_bwd, mask_f, mask_b, sort_f, sort_b, masks = res
    assert len(mask_f) == 2 and len(sort_f) == 2 and len(masks) == 2
    assert int(masks[0][0]) == (1 << 14) - 1 and int(masks[1][0]) == ((1 << 13) - 1) << 14
    o, pairs, num = oracle.get_indice_pairs(inds, 1, shape, k, s, p, [1] * 3, [0] * 3, subm)
    tabs = oracle.implicit_gemm_tables(pairs, num, inds.shape[0], o.shape[0], subm)
    full = tabs["mask_fwd_unsorted"][:, 0]
    for j in range(2):
        want = full & masks[j][0]
        order = np.argsort(want, kind="stable")
        assert np.array_equal(sort_f[j].cpu().numpy(), order)
        assert np.array_equal(mask_f[j].cpu().numpy().view(np.uint32)[:, 0], want[order])
    # module level: same weights, split vs unsplit
    cls = spconv.SubMConv3d if subm else spconv.SparseConv3d
    args = (32, 48, 3) if subm else (32, 48, 3, 2, 1)
    a = cls(*args, bias=True, algo=ConvAlgo.MaskImplicitGemm).to(cuda_dev).half()
    b = cls(*args, bias=True, algo=ConvAlgo.MaskSplitImplicitGemm).to(cuda_dev).half()
    b.load_state_dict(a.state_dict())
    outs = []
    for m in (a, b):
        xf = torch.from_numpy(feats).to(cuda_dev).half().requires_grad_(True)
        y = m(spconv.SparseConvTensor(xf, d_inds, shape, 1))
        (y.features.float().square().sum() * 1e-2).backward()       # keeps fp16 gradients out of the subnormals
        outs.append((y.features.detach().float(), xf.grad.float(), m.weight.grad.float(), m.bias.grad.float()))
    for u, v in zip(*outs):
        assert rel_l2(v.cpu().numpy(), u.cpu().numpy()) < 5e-3
    # inference path with fused bias + activation after the last split
    a.eval(), b.eval()
    a.act_type = b.act_type = spconv.Activation.ReLU
    with torch.no_grad():
        x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev).half(), d_inds, shape, 1)
        ya, yb = a(x).features.float(), b(x).features.float()
    assert (ya >= 0).all() and rel_l2(yb.cpu().numpy(), ya.cpu().numpy()) < 5e-3


@pytest.mark.parametrize("subm", [True, False])
def test_quantized_sparse_conv_hookup(subm, oracle, cuda_dev):
    """static int8 module: per-channel scale derivation of the reference
    (spconv/pytorch/quantization/quantized/conv.py:368-377) + the int8 kernel; exact against the
    numpy formula of test/test_all_algo.py:272-287, close to the float layer"""
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch import quantized as Q
    rng = np.random.default_rng(8)
    shape = [20, 20, 20]
    feats, inds = random_cloud(rng, shape, [2500], 32)
    cls, args = (spconv.SubMConv3d, (32, 64, 3)) if subm else (spconv.SparseConv3d, (32, 64, 3, 2, 1))
    fconv = cls(*args, bias=True).to(cuda_dev).eval()
    fconv.act_type = spconv.Activation.ReLU
    x = spconv.SparseConvTensor(torch.from_numpy(feats).to(cuda_dev), torch.from_numpy(inds).to(cuda_dev), shape, 1)
    out_scale = Q.calibrate_output_scale(fconv, x)
    qconv = Q.QuantizedSparseConv.from_float(fconv, out_scale)
    in_scale = 1.0 / 127.0
    xq = Q.quantize_tensor(x, in_scale)
    with torch.no_grad():
        yq = qconv(xq)
        yf = fconv(x)
    assert yq.features.dtype == torch.int8 and yq.int8_scale == out_scale
    # exact vs the reference formula
    s = [1] * 3 if subm else [2] * 3
    o, pairs, num = oracle.get_indice_pairs(inds, 1, shape, [3] * 3, s, [1] * 3, [1] * 3, [0] * 3, subm)
    ch_scale = (in_scale * qconv.weight_scales.cpu().numpy()) / out_scale
    ref = oracle.int8_conv_forward(xq.features.cpu().numpy(), qconv.weight.cpu().numpy(), pairs, num, o.shape[0], subm,
                                   ch_scale.astype(np.float32), (qconv.bias.cpu().numpy() / out_scale).astype(np.float32),
                                   relu=True, out_int8=True)
    got = yq.features.cpu().numpy()
    assert np.array_equal(yq.indices.cpu().numpy(), o)
    # rint at exact .5 ties can differ by fp32 evaluation order: allow a handful of off-by-one
    diff = np.abs(got.astype(np.int32) - ref.astype(np.int32))
    assert diff.max() <= 1 and (diff != 0).mean() < 1e-3, (diff.max(), (diff != 0).mean())
    # close to the float layer (quantisation noise only)
    deq = Q.dequantize_tensor(yq).features
    err = (deq - yf.features).abs().max() / yf.features.abs().max()
    assert float(err) < 0.05, float(err)


def test_graph_capture_of_a_subm_training_step(cuda_dev):
    """spconv.graph_capture: a SubM stack's forward + backward replayed as ONE CUDA graph gives the
    eager result bit for bit; a strided conv inside the captured region is refused with a clear error"""
    import spconv_b200.pytorch as spconv
    rng = np.random.default_rng(17)
    shape = [24, 24, 24]
    feats, inds = random_cloud(rng, shape, [3000], 32)
    net = spconv.SparseSequential(spconv.SubMConv3d(32, 32, 3, bias=False, indice_key="k"),
                                  spconv.SubMConv3d(32, 64, 3, bias=False, indice_key="k")).to(cuda_dev).half()
    d_inds = torch.from_numpy(inds).to(cuda_dev)
    params = list(net.parameters())

    def step(f, i):
        for p in params:
            p.grad = None
        y = net(spconv.SparseConvTensor(f, i, shape, 1))
        loss = y.features.float().square().mean()
        loss.backward()
        return loss, [p.grad for p in params]

    f0 = torch.from_numpy(feats).to(cuda_dev).half()
    loss_e, grads_e = step(f0, d_inds)
    # detach: a live autograd graph from an eager step keeps its AccumulateGrad nodes (bound to the
    # stream they were created on) alive, and a capture must not touch the legacy default stream
    loss_e, grads_e = loss_e.detach().clone(), [g.detach().clone() for g in grads_e]
    g = spconv.graph_capture(step, f0, d_inds)
    f1 = (f0 * 0.5).contiguous()
    g(f1, d_inds)                                        # different data, same shapes
    loss_g, grads_g = g(f0, d_inds)
    assert torch.equal(loss_g, loss_e)
    for a, b in zip(grads_g, grads_e):
        assert torch.equal(a, b)
    down = spconv.SparseConv3d(32, 32, 3, 2, 1, bias=False).to(cuda_dev).half()
    with pytest.raises(RuntimeError, match="cannot be captured"):
        spconv.graph_capture(lambda f, i: down(spconv.SparseConvTensor(f, i, shape, 1)).features, f0, d_inds)
    torch.cuda.synchronize()
    # the library is usable again after the refused capture
    y = down(spconv.SparseConvTensor(f0, d_inds, shape, 1))
    assert torch.isfinite(y.features.float()).all()


def test_rulebook_prefetch_on_a_side_stream(cuda_dev):
    """RulebookPrefetcher: the next batch's SubM rulebooks are built on a side stream and found by the
    layers through indice_key; results equal the unprefetched run and no rulebook kernel runs in forward"""
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch import ops
    rng = np.random.default_rng(23)
    shape = [24, 24, 24]
    feats, inds = random_cloud(rng, shape, [3000], 32)
    net = spconv.SparseSequential(spconv.SubMConv3d(32, 32, 3, bias=False, indice_key="a"),
                                  spconv.SubMConv3d(32, 64, 3, bias=False, indice_key="a"),
                                  spconv.SparseConv3d(64, 64, 3, 2, 1, bias=False),
                                  spconv.SubMConv3d(64, 64, 3, bias=False, indice_key="b")).to(cuda_dev).half()
    pre = spconv.RulebookPrefetcher(net)
    assert [m.indice_key for m in pre.layers] == ["a", "a"]      # the keyless strided layer ends the chain
    f = torch.from_numpy(feats).to(cuda_dev).half()
    i = torch.from_numpy(inds).to(cuda_dev)
    ref = net(spconv.SparseConvTensor(f, i, shape, 1))
    x = pre.prefetch(spconv.SparseConvTensor(f, i, shape, 1))
    assert "a" in x.indice_dict
    torch.cuda.synchronize()
    ops.launch_count(reset=True)
    y = net(pre.ready(x))
    n_prefetched = ops.launch_count(reset=True)
    ops.launch_count(reset=True)
    net(spconv.SparseConvTensor(f, i, shape, 1))
    n_plain = ops.launch_count(reset=True)
    assert torch.equal(y.features, ref.features) and torch.equal(y.indices, ref.indices)
    assert n_prefetched < n_plain                                  # the SubM "a" rulebook kernels are gone


def test_rulebook_prefetch_follows_strided_layers_from_a_worker_thread(cuda_dev):
    """Full-chain prefetch: every keyed layer's rulebook -- the strided ones too, whose output-count
    read-back then happens on the prefetch stream in a worker thread -- is built ahead; the forward pass
    launches no rulebook kernel, results and gradients equal the plain run; a strided layer refuses a
    cached rulebook that was not prefetched for its geometry."""
    import spconv_b200.pytorch as spconv
    from spconv_b200.pytorch import ops
    from bench_utils import make_encoder6
    rng = np.random.default_rng(29)
    shape = [32, 48, 40]
    feats, inds = random_cloud(rng, shape, [2500, 1800], 16)
    layers = [m.to(cuda_dev).half() for m in make_encoder6(spconv)]
    net = spconv.SparseSequential(*layers)
    pre = spconv.RulebookPrefetcher(net, background=True)
    assert [m.indice_key for m in pre.layers] == ["subm1", "subm1", "down1", "subm2", "down2", "down3"]
    i = torch.from_numpy(inds).to(cuda_dev)

    def run(x):
        for m in layers:
            m.weight.grad = None
        y = net(x)
        (y.features.float().square().mean() * 64).backward()
        return y, [m.weight.grad.clone() for m in layers], x.features.grad.clone()

    f = torch.from_numpy(feats).to(cuda_dev).half()
    y0, gw0, gx0 = run(spconv.SparseConvTensor(f.clone().requires_grad_(True), i, shape, 2))
    ops.launch_count(reset=True)
    run(spconv.SparseConvTensor(f.clone().requires_grad_(True), i, shape, 2))
    n_plain = ops.launch_count(reset=True)

    for _ in range(3):                                             # steady state: prefetch, then consume
        x = pre.prefetch(spconv.SparseConvTensor(f.clone().requires_grad_(True), i, shape, 2))
        x = pre.ready(x)
        assert set(x.indice_dict) == {"subm1", "down1", "subm2", "down2", "down3"}
        n_rulebook = ops.launch_count(reset=True)
        y1, gw1, gx1 = run(x)
        n_gemm = ops.launch_count(reset=True)
        assert torch.equal(y1.indices, y0.indices) and torch.equal(y1.features, y0.features)
        assert torch.equal(gx1, gx0) and all(torch.equal(a, b) for a, b in zip(gw1, gw0))
        assert n_rulebook > 0 and n_rulebook + n_gemm == n_plain   # same kernels, moved ahead of the step
    pre.shutdown()

    # a strided layer with somebody else's key: cached, but not prefetched for this geometry
    x = spconv.RulebookPrefetcher(net).prefetch(spconv.SparseConvTensor(f, i, shape, 2))
    other = spconv.SparseConv3d(16, 32, 3, stride=1, padding=1, bias=False, indice_key="down1").to(cuda_dev).half()
    with pytest.raises(ValueError, match="does not match this layer"):
        other(x)
