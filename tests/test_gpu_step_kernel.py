"""The one-kernel worker step (csrc/mlp_step.cu) on hardware: TMA-fed tcgen05.mma.kind::tf32 tiles, the L2 exchange between
its CTAs, the fused head and the pushed gradients, against a float64 PyTorch model of the reference network
(/root/reference/distributed_mnist.py:109-113) built from the UNROUNDED fp32 inputs.  Tolerances are TF32's (10-bit
mantissa on the two large GEMMs' operands); everything else is fp32."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _reference(x, y, w1, b1, w2, b2, clip=1e-10):
    d = lambda t: t.double()
    h = torch.relu(d(x) @ d(w1) + d(b1))
    z = h @ d(w2) + d(b2)
    p = torch.softmax(z, -1)
    loss = -(d(y) * torch.log(torch.clamp(p, clip, 1.0))).sum()
    keep = (p >= clip).double()
    dl = p * (d(y) * keep).sum(-1, keepdim=True) - d(y) * keep
    dh = (dl @ d(w2).t()) * (h > 0)
    return loss, z, {"w1": d(x).t() @ dh, "b1": dh.sum(0), "w2": h.t() @ dl, "b2": dl.sum(0), "dh": dh}


def _rel(a, b):
    return float((a.double().cpu() - b).norm() / (b.norm() + 1e-30))


def _check_backward(x, w1, b1, dh_k, gw1_k, gb1_k, ref, B, H):
    """dh carries the ReLU gate (h > 0): a pre-activation within TF32 rounding of zero may legitimately land on the other
    side, which flips that ONE element between d and 0 (a few per step; each is a full-magnitude difference).  So: dh is
    compared where the gate is unambiguous, and the two quantities computed FROM dh (dW1 = x^T.dh on the tensor cores,
    db1 = column sums) are checked against the kernel's own dh -- that isolates the GEMM / reduction being tested."""
    pre = x.double() @ w1.double() + b1.double()
    sure = pre.abs() > 1e-3 * (x.double().abs() @ w1.double().abs() + b1.double().abs())     # worst-case TF32 error of pre
    dh_k = dh_k[:B, :H].double().cpu()
    assert float(sure.double().mean()) > 0.9
    assert float(((dh_k - ref["dh"]) * sure).norm() / ref["dh"].norm()) < 3e-3
    assert int(((dh_k != 0) != (ref["dh"] != 0))[sure].sum()) == 0      # the gate itself agrees wherever it is unambiguous
    assert _rel(gw1_k, x.double().t() @ dh_k) < 2e-3
    assert _rel(gb1_k, dh_k.sum(0)) < 1e-5


@pytest.mark.parametrize("mask", [15, 7])            # 15: one launch per phase (no inter-CTA waits); 7: the fused kernel
@pytest.mark.parametrize("B,D,H,C,nbatches,wide", [(100, 784, 100, 10, 3, True), (100, 784, 100, 10, 3, False), (37, 200, 64, 7, 0, False),
                                                   (128, 96, 128, 16, 2, True)])
def test_step_kernel_matches_float64_model(B, D, H, C, nbatches, wide, mask):
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from distributed_tensorflow_b200.ops import cuda_lib
    lib = cuda_lib.load()
    dev = "cuda"
    g = torch.Generator().manual_seed(B + D)
    rows = max(nbatches, 1) * B
    xs_h = torch.rand(rows + 64, D, generator=g)                    # + slack rows: the 128-row box of the last batch
    ys_h = torch.nn.functional.one_hot(torch.randint(0, C, (rows,), generator=g), C).float()
    # wide: 128-float rows (the engine's tf32 layout: in-bounds TMA boxes, dW1 leaves as ONE bulk store per CTA)
    ldw1, ldw2 = (128 if wide else (H + 7) // 8 * 8), (C + 7) // 8 * 8
    w1_h = torch.zeros(D, ldw1); w1_h[:, :H] = torch.randn(D, H, generator=g) / np.sqrt(D)
    w2_h = torch.zeros(H, ldw2); w2_h[:, :C] = torch.randn(H, C, generator=g) / np.sqrt(H)
    b1_h, b2_h = torch.randn(H, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    xs, ys, w1, w2, b1, b2 = (t.to(dev) for t in (xs_h, ys_h, w1_h, w2_h, b1_h, b2_h))
    ds = ctypes.c_int(0)
    G = lib.dtf_mlp_step_slices(D, B, ctypes.byref(ds))
    n1 = (H + 15) // 16 * 16
    hpart = torch.zeros(G * 128 * (n1 + 4), device=dev)
    dh = torch.zeros(128, 128, device=dev)
    head_part = torch.zeros(G * lib.dtf_mlp_step_head_part_floats(), device=dev)
    flags = torch.zeros(8, dtype=torch.int32, device=dev)
    # every gradient is STORED: stale content of the slot must be overwritten
    gw1, gb1 = torch.full((D, ldw1), 7.0, device=dev), torch.full((H,), 7.0, device=dev)
    gw2, gb2 = torch.full((H, ldw2), 7.0, device=dev), torch.full((C,), 7.0, device=dev)
    loss, logits = torch.zeros(16, device=dev), torch.zeros(B, C, device=dev)
    step0 = 1 if nbatches else 0
    stepctr = torch.tensor([step0], dtype=torch.int64, device=dev)
    flags[:3] = G * 3
    flags[3] = 3
    token = torch.tensor([5, 9], dtype=torch.int64, device=dev)
    arrivals = torch.zeros(2, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    trace = torch.zeros(16 * 32, dtype=torch.int64, device=dev)
    p = lambda t: t.data_ptr()
    a = cuda_lib.MlpStepArgs()
    a.B, a.D, a.H, a.C, a.G, a.phase_mask = B, D, H, C, 0, mask
    a.x, a.ldx, a.x_rows = p(xs), D, rows + 64
    a.labels, a.ldl = p(ys), C
    a.nbatches, a.bstride, a.boffset = nbatches, 2, 1
    a.w1, a.ldw1, a.b1, a.w2, a.ldw2, a.b2 = p(w1), ldw1, p(b1), p(w2), ldw2, p(b2)
    a.hpart, a.dh, a.lddh, a.flags = p(hpart), p(dh), 128, p(flags)
    a.gw1, a.ldgw1, a.gb1, a.gw2, a.ldgw2, a.gb2 = p(gw1), ldw1, p(gb1), p(gw2), ldw2, p(gb2)
    a.head_part = p(head_part)
    a.clip_min, a.loss_out, a.logits_out, a.step_counter = 1e-10, p(loss), p(logits), p(stepctr)
    a.num_tokens, a.token[0] = 1, p(token)
    a.num_signals, a.arrivals[0], a.stamp_dst[0], a.stamp_src[0] = 1, p(arrivals), p(arrivals) + 8, p(token)
    a.sys_scope, a.timeout_ns, a.err, a.trace = 1, 2 * 10**9, p(err), p(trace)
    rc = lib.dtf_mlp_step(ctypes.byref(a), torch.cuda.current_stream().cuda_stream)
    assert rc == 0, rc
    torch.cuda.synchronize()
    assert int(err[0]) == 0
    bi = ((step0 * 2 + 1) % nbatches) if nbatches else 0
    x, y = xs_h[bi * B:(bi + 1) * B], ys_h[bi * B:(bi + 1) * B]
    ref_loss, ref_z, ref = _reference(x, y, w1_h[:, :H], b1_h, w2_h[:, :C], b2_h)
    assert _rel(logits, ref_z) < 2e-3
    assert abs(float(loss[:G].sum()) - float(ref_loss)) < 2e-3 * abs(float(ref_loss))
    _check_backward(x, w1_h[:, :H], b1_h, dh, gw1[:, :H], gb1, ref, B, H)
    assert float(dh[B:].abs().sum()) == 0.0 and float(dh[:, H:].abs().sum()) == 0.0
    assert _rel(gw2[:, :C], ref["w2"]) < 3e-3 and _rel(gb2, ref["b2"]) < 3e-3
    assert int(stepctr[0]) == step0 + 1
    assert int(arrivals[0]) == G and int(arrivals[1]) == 5
    clustered = mask == 7 and G <= 8                               # one cluster: barrier.cluster instead of the two L2 counters
    assert flags[:4].tolist() == [G * (3 if clustered else 4)] * 2 + [G * 4, 4] and flags[4:].tolist() == [0] * 4
    if wide:
        assert float(gw1[:, H:].abs().sum()) == 0.0                # padding columns of the slot receive exact zeros
    if mask == 7:
        t = trace.view(16, 32)[:G].cpu()
        assert bool((t[:, 10] > t[:, 0]).all())                    # every CTA stamped entry and exit


def test_step_kernel_two_consecutive_steps_and_forward_only():
    """The counters are monotonic (G per step): a second launch walks to the next batch; a forward-only launch (validation /
    predict) returns loss + logits and touches neither the gradients nor the protocol."""
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    from distributed_tensorflow_b200.ops import cuda_lib
    lib = cuda_lib.load()
    dev = "cuda"
    B, D, H, C, nb = 100, 784, 100, 10, 4
    g = torch.Generator().manual_seed(0)
    xs_h = torch.rand(nb * B + 64, D, generator=g)
    ys_h = torch.nn.functional.one_hot(torch.randint(0, C, (nb * B,), generator=g), C).float()
    w1_h = torch.zeros(D, 104); w1_h[:, :H] = torch.randn(D, H, generator=g) / 28
    w2_h = torch.zeros(H, 16); w2_h[:, :C] = torch.randn(H, C, generator=g) / 10
    xs, ys, w1, w2 = xs_h.to(dev), ys_h.to(dev), w1_h.to(dev), w2_h.to(dev)
    b1, b2 = torch.zeros(H, device=dev), torch.zeros(C, device=dev)
    G = lib.dtf_mlp_step_slices(D, B, None)
    hpart, dh = torch.zeros(G * 128 * 116, device=dev), torch.zeros(128, 128, device=dev)
    head_part = torch.zeros(G * lib.dtf_mlp_step_head_part_floats(), device=dev)
    flags = torch.zeros(8, dtype=torch.int32, device=dev)
    gw1, gb1, gw2, gb2 = (torch.zeros(s, device=dev) for s in ((D, 104), (H,), (H, 16), (C,)))
    loss, logits = torch.zeros(16, device=dev), torch.zeros(B, C, device=dev)
    stepctr = torch.zeros(1, dtype=torch.int64, device=dev)
    token = torch.tensor([1, 1], dtype=torch.int64, device=dev)
    arrivals = torch.zeros(2, dtype=torch.int64, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    p = lambda t: t.data_ptr()
    a = cuda_lib.MlpStepArgs()
    a.B, a.D, a.H, a.C, a.phase_mask = B, D, H, C, 7
    a.x, a.ldx, a.x_rows, a.labels, a.ldl = p(xs), D, nb * B + 64, p(ys), C
    a.nbatches, a.bstride, a.boffset = nb, 1, 0
    a.w1, a.ldw1, a.b1, a.w2, a.ldw2, a.b2 = p(w1), 104, p(b1), p(w2), 16, p(b2)
    a.hpart, a.dh, a.lddh, a.flags = p(hpart), p(dh), 128, p(flags)
    a.gw1, a.ldgw1, a.gb1, a.gw2, a.ldgw2, a.gb2 = p(gw1), 104, p(gb1), p(gw2), 16, p(gb2)
    a.head_part = p(head_part)
    a.clip_min, a.loss_out, a.logits_out, a.step_counter = 1e-10, p(loss), p(logits), p(stepctr)
    a.num_tokens, a.token[0] = 1, p(token)
    a.num_signals, a.arrivals[0], a.stamp_dst[0], a.stamp_src[0] = 1, p(arrivals), p(arrivals) + 8, p(token)
    a.sys_scope, a.timeout_ns, a.err = 0, 2 * 10**9, p(err)
    st = torch.cuda.current_stream().cuda_stream
    for t in range(2):
        gw2.fill_(7.0); gb2.fill_(7.0); gb1.fill_(7.0)              # the step overwrites what the previous one left
        assert lib.dtf_mlp_step(ctypes.byref(a), st) == 0
        torch.cuda.synchronize()
        ref_loss, _, ref = _reference(xs_h[t * B:(t + 1) * B], ys_h[t * B:(t + 1) * B], w1_h[:, :H], b1.cpu(), w2_h[:, :C], b2.cpu())
        assert abs(float(loss[:G].sum()) - float(ref_loss)) < 2e-3 * abs(float(ref_loss))
        _check_backward(xs_h[t * B:(t + 1) * B], w1_h[:, :H], b1.cpu(), dh, gw1[:, :H], gb1, ref, B, H)
    assert int(stepctr[0]) == 2 and int(arrivals[0]) == 2 * G and int(err[0]) == 0
    # forward-only on batch 2 (the step counter selects it and is NOT advanced)
    before = (gw1.clone(), int(arrivals[0]))
    a.forward_only, a.phase_mask = 1, 7
    assert lib.dtf_mlp_step(ctypes.byref(a), st) == 0
    torch.cuda.synchronize()
    ref_loss, ref_z, _ = _reference(xs_h[2 * B:3 * B], ys_h[2 * B:3 * B], w1_h[:, :H], b1.cpu(), w2_h[:, :C], b2.cpu())
    assert _rel(logits, ref_z) < 2e-3
    assert abs(float(loss[:G].sum()) - float(ref_loss)) < 2e-3 * abs(float(ref_loss))
    assert torch.equal(before[0], gw1) and int(arrivals[0]) == before[1] and int(stepctr[0]) == 2
    assert flags.tolist() == [0, 0, 2 * G, 2, 0, 0, G, 1]           # clustered launches: only the ticket + epoch counters move
