"""GPU: the logit KD op right behind a kernel that writes its inputs.

The row kernel asks L2 for its operand rows before its programmatic dependency wait, while the predecessor may still be
writing them, and a second launch folds the row partials into the loss.  A CUDA graph of steps in which a copy kernel
refills the op's inputs immediately before each forward + backward must give, bit for bit, the losses and gradients of
eager steps in which a synchronisation separates the copy from the op."""
import pytest
import torch

from deltakd_b200 import functional as Fn, synth

pytestmark = pytest.mark.gpu


def _fwd_bwd(x):
    z = x[0].detach().requires_grad_(True)
    zk = x[1].detach().requires_grad_(True)
    loss = Fn.logit_kd_loss(z, zk, x[2], x[3], kd_kind="soft", alpha=0.1, tau=3.0)
    loss.backward()
    return loss.detach(), z.grad, zk.grad


@pytest.mark.parametrize("B,C,dtype", [
    (8, 1000, torch.float32),      # few row CTAs
    (256, 1000, torch.bfloat16),   # the headline shape
    (37, 1001, torch.bfloat16),    # rows not 16-byte aligned: per-line prefetches, streaming kernel
    (1025, 104, torch.bfloat16),   # B >= 1024 with rows too short for the bulk-copy ring: 1024-thread fold
])
def test_graph_with_input_writer_before_each_call_matches_eager(B, C, dtype):
    steps = 3
    # float64 sources: copy_ into the op's dtype is a conversion kernel (not a memcpy) writing all four operands
    src = [torch.empty(4, B, C, dtype=torch.float64, device="cuda") for _ in range(steps)]
    static = torch.empty(4, B, C, dtype=dtype, device="cuda")

    def fill(rot):
        for k in range(steps):
            src[k].copy_(torch.stack(synth.make_logits(B, C, 1000 * rot + 31 * k + B)).double())

    def run():
        outs = []
        for k in range(steps):
            static.copy_(src[k])
            outs.append(tuple(t.clone() for t in _fwd_bwd(static)))
        return outs

    fill(0)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()   # warm-up on the capture stream (its workspace is cached there)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        outs = run()
    for rot in range(2):
        fill(rot)
        want = []
        for k in range(steps):
            static.copy_(src[k])
            torch.cuda.synchronize()
            want.append(_fwd_bwd(static))
            torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        for k in range(steps):
            assert torch.isfinite(want[k][0])
            for got, ref in zip(outs[k], want[k]):
                assert torch.equal(got, ref), (rot, k)
