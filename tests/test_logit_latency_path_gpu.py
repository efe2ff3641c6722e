"""GPU: the small-batch logit KD path (one CTA per row, partials published before the gradient stores, last CTA folds)
and its programmatic dependent launches (the logit kernel and the gradient rescale start while their predecessor runs).

Determinism across runs, CUDA-graph capture of consecutive steps against eager steps, and back-to-back calls on one
stream and one workspace against calls separated by a synchronisation."""
import pytest
import torch

from deltakd_b200 import functional as Fn, synth

pytestmark = pytest.mark.gpu

C = 1000


def _inputs(B, dtype, seed, int_labels=False):
    z, zk, zt, y = synth.make_logits(B, C, seed, int_labels=int_labels)
    cast = lambda t: t.to(dtype).cuda()
    return cast(z), cast(zk), cast(zt), (y.cuda() if int_labels else cast(y))


def _fwd_bwd(z, zk, zt, y, kind, grad_output=None):
    z = z.detach().requires_grad_(True)
    zk = zk.detach().requires_grad_(True)
    loss = Fn.logit_kd_loss(z, zk, zt, y, kd_kind=kind, alpha=0.1, tau=3.0)
    loss.backward(grad_output)
    return loss.detach(), z.grad, zk.grad


@pytest.mark.parametrize("kind", ["soft", "hard"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("B", [1, 8, 255, 256, 257, 1023])
def test_two_runs_are_bit_identical(B, dtype, kind):
    ins = _inputs(B, dtype, 100 + B)
    a = _fwd_bwd(*ins, kind)
    b = _fwd_bwd(*ins, kind)
    torch.cuda.synchronize()
    assert torch.isfinite(a[0]) and torch.isfinite(a[1].float()).all() and torch.isfinite(a[2].float()).all()
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.parametrize("go", [1.0, 0.5])
def test_graph_of_three_steps_replays_like_eager(go):
    """Three forward + backward steps captured in one graph (each step's kernels follow the previous step's through
    programmatic edges); replayed on two rotations of the inputs, every loss and gradient equals the eager step's."""
    B, steps = 256, 3
    static = [[torch.empty(B, C, dtype=torch.bfloat16, device="cuda") for _ in range(4)] for _ in range(steps)]
    g_out = torch.full((), go, dtype=torch.float32, device="cuda")

    def fill(rot):
        for i in range(steps):
            for dst, src in zip(static[i], _inputs(B, torch.bfloat16, 7 + 10 * rot + i)):
                dst.copy_(src)

    def run():
        return [tuple(t.clone() for t in _fwd_bwd(*static[i], "soft", g_out)) for i in range(steps)]

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
        torch.cuda.synchronize()
        want = run()
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        for i in range(steps):
            for got, ref in zip(outs[i], want[i]):
                assert torch.equal(got, ref), (rot, i)
        assert go == 1.0 or not torch.equal(outs[0][1], _fwd_bwd(*static[0], "soft")[1])   # the rescale did run


@pytest.mark.parametrize("dtype,B", [(torch.bfloat16, 256), (torch.float32, 8), (torch.float32, 256)])
def test_back_to_back_calls_match_separate_calls(dtype, B):
    """K op calls queued on one stream (one workspace, one ticket) without a host synchronisation between them give the
    results of the same calls separated by synchronisations."""
    K = 16
    sets = [_inputs(B, dtype, 500 + k) for k in range(K)]
    want = []
    for s in sets:
        want.append(_fwd_bwd(*s, "soft"))
        torch.cuda.synchronize()
    got = [_fwd_bwd(*s, "soft") for s in sets]
    torch.cuda.synchronize()
    for g, w in zip(got, want):
        for x, y in zip(g, w):
            assert torch.equal(x, y)
