"""The one-kernel worker step (csrc/mlp_step.cu) under the host emulation: same source, the TMA / tcgen05 parts replaced by
scalar loops, the three phases launched one after another (emulated blocks run sequentially).  Checks everything around the
tensor-core tiles -- slice / row ownership, the L2 exchange buffers, the fused head (softmax, clipped batch-SUM
cross-entropy, dlogits, dh, dW2 / db2 / db1 partial sums added in CTA order), the dW1 store pattern, the device step counter,
stamp + arrival -- against a float64 PyTorch model of /root/reference/distributed_mnist.py:109-113."""
import ctypes
import shutil

import numpy as np
import pytest
import torch

from distributed_tensorflow_b200.ops import cuda_lib


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("g++ not available")
    lib = cuda_lib.enable_emulation(str(tmp_path_factory.mktemp("emu_step")))
    yield lib
    cuda_lib.disable_emulation()


def _ptr(t):
    return t.data_ptr()


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


@pytest.mark.parametrize("B,D,H,C,nbatches", [(100, 784, 100, 10, 3), (37, 200, 64, 7, 0), (128, 96, 128, 16, 2), (128, 24, 32, 3, 0)])
def test_step_kernel_matches_float64_model(emu, B, D, H, C, nbatches):
    g = torch.Generator().manual_seed(B + D)
    rows = max(nbatches, 1) * B
    xs = torch.rand(rows, D, generator=g)
    ys = torch.nn.functional.one_hot(torch.randint(0, C, (rows,), generator=g), C).float()
    ldw1, ldw2 = (H + 7) // 8 * 8, (C + 7) // 8 * 8
    w1 = torch.zeros(D, ldw1); w1[:, :H] = torch.randn(D, H, generator=g) / np.sqrt(D)
    w2 = torch.zeros(H, ldw2); w2[:, :C] = torch.randn(H, C, generator=g) / np.sqrt(H)
    b1, b2 = torch.randn(H, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    ds = ctypes.c_int(0)
    G = emu.dtf_mlp_step_slices(D, B, ctypes.byref(ds))
    assert G * ds.value >= D and ds.value % 8 == 0 and (B + G - 1) // G <= 16
    if D == 784:
        assert (G, ds.value) == (7, 112)
    n1 = (H + 15) // 16 * 16
    hpart = torch.zeros(G * 128 * (n1 + 4))
    dh = torch.zeros(128, 128)
    head_part = torch.zeros(G * emu.dtf_mlp_step_head_part_floats())
    flags = torch.zeros(8, dtype=torch.int32)
    # every gradient is STORED (stale content must be overwritten); the head's sums in a fixed order of the CTA partials
    gw1, gb1 = torch.full((D, ldw1), 7.0), torch.full((H,), 7.0)
    gw2, gb2 = torch.full((H, ldw2), 7.0), torch.full((C,), 7.0)
    loss = torch.zeros(16)
    logits = torch.zeros(B, C)
    stepctr = torch.tensor([1 if nbatches else 0], dtype=torch.int64)
    token = torch.tensor([5, 9], dtype=torch.int64)                # mailbox {token, version}: already ahead of the step
    arrivals = torch.zeros(2, dtype=torch.int64)                   # {arrivals, stamp}
    err = torch.zeros(1, dtype=torch.int32)
    a = cuda_lib.MlpStepArgs()
    a.B, a.D, a.H, a.C, a.G, a.phase_mask = B, D, H, C, 0, 7
    a.x, a.ldx, a.x_rows = _ptr(xs), D, rows
    a.labels, a.ldl = _ptr(ys), C
    a.nbatches, a.bstride, a.boffset = nbatches, 2, 1
    a.w1, a.ldw1, a.b1, a.w2, a.ldw2, a.b2 = _ptr(w1), ldw1, _ptr(b1), _ptr(w2), ldw2, _ptr(b2)
    a.hpart, a.dh, a.lddh, a.flags = _ptr(hpart), _ptr(dh), 128, _ptr(flags)
    a.gw1, a.ldgw1, a.gb1, a.gw2, a.ldgw2, a.gb2 = _ptr(gw1), ldw1, _ptr(gb1), _ptr(gw2), ldw2, _ptr(gb2)
    a.head_part = _ptr(head_part)
    a.clip_min, a.loss_out, a.logits_out, a.step_counter = 1e-10, _ptr(loss), _ptr(logits), _ptr(stepctr)
    a.num_tokens, a.token[0] = 1, _ptr(token)
    a.num_signals, a.arrivals[0], a.stamp_dst[0], a.stamp_src[0] = 1, _ptr(arrivals), _ptr(arrivals) + 8, _ptr(token)
    a.sys_scope, a.timeout_ns, a.err = 1, 10**9, _ptr(err)
    step0 = int(stepctr[0])
    flags[:3] = G * 3                                              # counters are monotonic: as if three launches ran before
    flags[3] = 3
    assert emu.dtf_mlp_step(ctypes.byref(a), None) == 0
    bi = ((step0 * 2 + 1) % nbatches) if nbatches else 0
    x, y = xs[bi * B:(bi + 1) * B], ys[bi * B:(bi + 1) * B]
    ref_loss, ref_z, ref = _reference(x, y, w1[:, :H], b1, w2[:, :C], b2)
    assert int(err[0]) == 0
    assert abs(float(loss[:G].sum()) - float(ref_loss)) < 1e-4 * abs(float(ref_loss))
    torch.testing.assert_close(logits.double(), ref_z, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(dh[:B, :H].double(), ref["dh"], rtol=1e-4, atol=1e-6)
    assert float(dh[B:].abs().sum()) == 0.0 and float(dh[:, H:].abs().sum()) == 0.0       # the padding the B3 GEMM relies on
    torch.testing.assert_close(gw1[:, :H].double(), ref["w1"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gb1.double(), ref["b1"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gw2[:, :C].double(), ref["w2"], rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(gb2.double(), ref["b2"], rtol=1e-4, atol=1e-5)
    assert int(stepctr[0]) == step0 + 1                            # CTA 0 advanced the device step counter once
    assert int(arrivals[0]) == G and int(arrivals[1]) == 5         # one arrival per CTA, stamp = the token
    assert flags[:4].tolist() == [G * 4] * 3 + [4] and flags[4:].tolist() == [0] * 4


def test_forward_only_leaves_gradients_and_protocol_untouched(emu):
    B, D, H, C = 100, 784, 100, 10
    g = torch.Generator().manual_seed(3)
    x = torch.rand(B, D, generator=g)
    y = torch.nn.functional.one_hot(torch.randint(0, C, (B,), generator=g), C).float()
    w1, w2 = torch.randn(D, 104, generator=g) / 28, torch.randn(H, 16, generator=g) / 10
    b1, b2 = torch.zeros(H), torch.zeros(C)
    G = emu.dtf_mlp_step_slices(D, B, None)
    hpart, dh, flags = torch.zeros(G * 128 * 116), torch.zeros(128, 128), torch.zeros(8, dtype=torch.int32)
    loss, logits = torch.zeros(16), torch.zeros(B, C)
    stepctr, token = torch.zeros(1, dtype=torch.int64), torch.zeros(2, dtype=torch.int64)
    arrivals = torch.zeros(2, dtype=torch.int64)
    a = cuda_lib.MlpStepArgs()
    a.B, a.D, a.H, a.C, a.phase_mask, a.forward_only = B, D, H, C, 3, 1
    a.x, a.ldx, a.x_rows, a.labels, a.ldl = _ptr(x), D, B, _ptr(y), C
    a.w1, a.ldw1, a.b1, a.w2, a.ldw2, a.b2 = _ptr(w1), 104, _ptr(b1), _ptr(w2), 16, _ptr(b2)
    a.hpart, a.dh, a.lddh, a.flags = _ptr(hpart), _ptr(dh), 128, _ptr(flags)
    a.clip_min, a.loss_out, a.logits_out, a.step_counter = 1e-10, _ptr(loss), _ptr(logits), _ptr(stepctr)
    a.num_tokens, a.token[0] = 1, _ptr(token)
    a.num_signals, a.arrivals[0] = 1, _ptr(arrivals)
    a.timeout_ns = 10**9
    assert emu.dtf_mlp_step(ctypes.byref(a), None) == 0
    ref_loss, ref_z, _ = _reference(x, y, w1[:, :H], b1, w2[:, :C], b2)
    assert abs(float(loss[:G].sum()) - float(ref_loss)) < 1e-4 * abs(float(ref_loss))
    torch.testing.assert_close(logits.double(), ref_z, rtol=1e-4, atol=1e-5)
    assert int(stepctr[0]) == 0 and int(arrivals[0]) == 0 and float(dh.abs().max()) == 0.0
    assert flags.tolist() == [0, 0, 0, 0, G, 0, G, 1]              # forward-only launches keep their own counters
