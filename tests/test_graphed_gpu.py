"""The training step as CUDA-graph replays (leak_det_gnn_b200/graphed.py; reference step models/train_detector.py:302-317)
and the device-resident dropout seed it rests on (ltgnn_seed_source, include/ltgnn.h)."""
import pytest
import torch

from conftest import TOPO

pytestmark = pytest.mark.gpu


def _model(g, n_pipes, dropout, seed=42):
    from leak_det_gnn_b200.graph import parse_epanet_inp
    from leak_det_gnn_b200.models import LeakDetector

    pipes = [ln.split()[0] for ln in parse_epanet_inp(TOPO["LTA"])["PIPES"]][:n_pipes]
    torch.manual_seed(seed)
    return LeakDetector(TOPO["LTA"], [str(s) for s in g["sensor_node_ids"]], pipes, dropout=dropout).cuda().train()


def _batches(n, bsz, seg, n_s, n_cls, seed=5):
    gen = torch.Generator().manual_seed(seed)
    return [(torch.randn(bsz, seg, n_s, generator=gen), torch.randn(bsz, seg, 9, generator=gen),
             torch.randint(0, n_cls, (bsz,), generator=gen)) for _ in range(n)]


def test_seed_source_adds_to_the_seed_argument(graph_golden):
    """drop_seed = s with the device word holding k draws exactly the masks of drop_seed = s + k with no source:
    node init, fused layer, fused aggregation and the pipe head."""
    from leak_det_gnn_b200 import ops

    m = _model(graph_golden("LTA"), 20, 0.1)
    dev = torch.device("cuda")
    slot, _, ends32, inc = m._index_tensors(dev)
    h_s = torch.randn(3, 29, 64, device=dev)
    word = torch.tensor([1000], dtype=torch.int64, device=dev)
    lin1, lin2 = m.edge_head.mlp[0], m.edge_head.mlp[3]

    def run(seed):
        x0 = ops.node_init_fwd(h_s, slot, 661, m.sensor_to_node.weight, m.sensor_to_node.bias, 0.1, seed)
        x1 = ops.gcn_layer_fwd(m.pipe_graph, x0, m.convs[0].lin.weight, bias=m.convs[0].bias, relu=True, drop_p=0.1,
                               drop_seed=seed + 1)
        x2 = ops.spmm_fused(m.pipe_graph, x1, bias=m.convs[1].bias, relu=True, drop_p=0.1, drop_seed=seed + 2)
        torch.manual_seed(seed)        # ops.heads draws its own drop_seed from torch's CPU generator
        with torch.no_grad():
            part, _ = ops.heads(x2, ends32, lin1.weight, lin1.bias, lin2.weight, 0.1, True, inc)
        return x0, x1, x2, part

    with ops.device_seed(word):
        with_word = run(7)
    torch.cuda.synchronize()
    plain_same = run(7)
    for a, b in zip(with_word[:3], plain_same[:3]):
        assert not torch.equal(a, b), "the device word must change the masks"
    word.fill_(0)
    with ops.device_seed(word):
        zero_word = run(7)
    for a, b in zip(zero_word, plain_same):
        assert torch.equal(a, b)
    # s + k without a source == s with the word k (the head's seed is drawn inside ops.heads: compare the three others)
    shifted = run(1007)
    for a, b in zip(with_word[:3], shifted[:3]):
        assert torch.equal(a, b)


@pytest.mark.parametrize("with_predictor", [False, True])
def test_graphed_step_equals_eager_step(graph_golden, with_predictor):
    """Three replays from the same start as three eager steps (dropout off, so the only difference is the launch
    mechanism): identical losses and parameters, bit for bit -- every kernel is deterministic."""
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.models import NormalPredictorTCN, build_residual_sequence_from_segment
    from leak_det_gnn_b200.parallel import FlatGradBucket

    g = graph_golden("LTA")
    bsz, l_pred, l_det, n_pipes = 16, 36, 12, 24
    seg = l_det + (l_pred if with_predictor else 0)
    data = _batches(3, bsz, seg, 29, n_pipes + 1)
    torch.manual_seed(3)
    predictor = NormalPredictorTCN(29, 9).cuda().eval() if with_predictor else None

    def fresh():
        m = _model(g, n_pipes, 0.0)
        return m, FlatGradBucket(m.parameters()), torch.optim.AdamW(m.parameters(), lr=1e-3, weight_decay=1e-4, capturable=True)

    m_e, bucket_e, opt_e = fresh()
    losses_e = []
    for noisy, tf, label in data:
        noisy, tf, label = noisy.cuda(), tf.cuda(), label.cuda()
        if with_predictor:
            with torch.no_grad():
                residual = build_residual_sequence_from_segment(predictor, noisy, tf, l_pred, l_det)
            tf = tf[:, l_pred:, :].contiguous()
        else:
            residual = noisy
        bucket_e.zero()
        loss = torch.nn.functional.cross_entropy(m_e(residual, tf), label)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(m_e.parameters(), 1.0)
        opt_e.step()
        losses_e.append(loss.item())

    m_g, bucket_g, opt_g = fresh()
    step = GraphedTrainStep(m_g, opt_g, bucket_g, bsz, l_det, predictor=predictor, l_pred=l_pred if with_predictor else 0,
                            grad_clip=1.0)
    assert step.kernels_per_replay >= 15
    losses_g = [step(*b).item() for b in data]
    assert losses_g == losses_e, (losses_g, losses_e)
    for (n, a), b in zip(m_e.named_parameters(), m_g.parameters()):
        assert torch.equal(a, b), n
    assert all(float(st["step"]) == 3 for st in opt_g.state.values())


def test_graphed_step_draws_fresh_dropout_masks(graph_golden):
    """Train mode, p = 0.1, lr = 0: replays on the same batch give different losses (new masks every replay), and the
    same torch seed reproduces the sequence."""
    from leak_det_gnn_b200.graphed import GraphedTrainStep
    from leak_det_gnn_b200.parallel import FlatGradBucket

    g = graph_golden("LTA")
    batch = _batches(1, 16, 12, 29, 25)[0]

    def losses():
        m = _model(g, 24, 0.1)
        torch.manual_seed(11)
        step = GraphedTrainStep(m, None, FlatGradBucket(m.parameters()), 16, 12)
        return [step(*batch).item() for _ in range(4)]

    a, b = losses(), losses()
    assert len(set(a)) == 4, a
    assert a == b



def test_capture_keeps_the_cycle_collector_out():
    """ops.capture (used by the graphed steps and the explainer) finalises dead cycles before capturing -- here one
    holding a captured CUDA graph, whose destruction is not permitted during a capture -- and runs no collection
    until the capture has ended."""
    import gc
    import weakref

    from leak_det_gnn_b200 import ops

    class Holder:
        pass

    x = torch.arange(8.0, device="cuda")
    dead = Holder()
    dead.graph = torch.cuda.CUDAGraph()
    with ops.capture(dead.graph):
        x.add_(1.0)
    dead.cycle = dead
    gone = weakref.ref(dead)
    del dead
    cg = torch.cuda.CUDAGraph()
    with ops.capture(cg):
        state = (gone() is None, gc.isenabled())
        y = x * 2
    assert state == (True, False) and gc.isenabled()
    x.fill_(3.0)
    cg.replay()
    torch.cuda.synchronize()
    assert torch.equal(y, torch.full_like(x, 6.0))


def test_pipe_graph_finalised_during_a_capture_is_released_after_it():
    """A PipeGraph finalised inside a caller's own capture keeps its device arrays until no capture is underway:
    cudaFree is not permitted during a capture and would invalidate it."""
    import gc

    from leak_det_gnn_b200 import ops

    dev = torch.device("cuda")
    dead = ops.PipeGraph(torch.tensor([[0, 1], [1, 0]]), 2)
    hv = dead.handle(dev).value
    x = torch.arange(8.0, device=dev)
    gc.collect()
    cg = torch.cuda.CUDAGraph()
    with torch.cuda.graph(cg):
        y = x * 2
        del dead                         # finalised here, by reference count
        parked = [h.value for h in ops._RETIRED]
    x.fill_(3.0)
    cg.replay()
    torch.cuda.synchronize()
    assert hv in parked and torch.equal(y, torch.full_like(x, 6.0))
    live = ops.PipeGraph(torch.tensor([[0, 1], [1, 0]]), 2)
    live.handle(dev)                     # the next handle, outside any capture, releases the parked one
    assert not ops._RETIRED
