"""CPU tests of the host layer: module API / state-dict compatibility, RNG side effects, error behaviour, schedule
construction, pool and damage host logic (kernels are not launched; the step is stubbed where noted)."""
import random

import numpy as np
import pytest
import torch

from conftest import load_golden, load_params
import graph_neural_cellular_automata_b200 as G
from graph_neural_cellular_automata_b200.modules import _base
from graph_neural_cellular_automata_b200.modules.graph_augmentation import build_offsets


def test_state_dict_keys_match_reference_and_checkpoints_load():
    f = load_golden("facts.npz")
    g = G.NeuralCAGraph(16, graph_zero_padded_shift=False)
    c = G.NeuralCA(16)
    assert sorted(g.state_dict().keys()) == list(f["graph_keys"])
    assert sorted(c.state_dict().keys()) == list(f["classic_keys"])
    missing, unexpected = g.load_state_dict(load_params("weights_graph_ep960.npz"), strict=True)
    assert not missing and not unexpected
    c.load_state_dict(load_params("weights_classic_ep990.npz"), strict=True)
    assert sum(p.numel() for p in g.parameters()) == 11185
    assert sum(p.numel() for p in g.parameters() if p.requires_grad) == 10753
    assert sum(p.numel() for p in c.parameters()) == 8784
    assert not g.perception.conv.weight.requires_grad


def test_offsets_and_attributes():
    f = load_golden("facts.npz")
    g = G.GraphAugmentation(16)
    assert g.offsets == [tuple(int(v) for v in o) for o in f["offsets_r4"]] and len(g.offsets) == 72
    assert build_offsets(2) == [tuple(int(v) for v in o) for o in f["offsets_r2"]]
    assert g.zero_padded_shift is True and g.alive_to_alive is True and g.num_neighbors == 8
    assert float(g.scaling.detach()) == pytest.approx(4.0)
    m = G.NeuralCAGraph(16, alpha_thr=0.12, message_gain=0.3)
    assert m.graph.alpha_thr == pytest.approx(0.12) and m.message_gain == pytest.approx(0.3) and m.hidden_only


def test_seeded_init_matches_reference_layer_order():
    """Same layer types created in the same order => same init as the reference under a seed (weights fixture
    was produced by the reference's ctor + checkpoint, so compare two of our own constructions for determinism
    and the zero-init of the last conv)."""
    torch.manual_seed(5); a = G.NeuralCAGraph(16)
    torch.manual_seed(5); b = G.NeuralCAGraph(16)
    for (ka, va), (kb, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        assert ka == kb and torch.equal(va, vb)
    assert float(a.update_net[2].weight.abs().sum()) == 0.0
    w = a.perception.conv.weight
    assert torch.equal(w[0, 0], torch.tensor([[0., 0, 0], [0, 1, 0], [0, 0, 0]]))
    assert torch.equal(w[1, 0], torch.tensor([[1., 0, -1], [2, 0, -2], [1, 0, -1]]))
    assert torch.equal(w[2, 0], torch.tensor([[1., 2, 1], [0, 0, 0], [-1, -2, -1]]))


def test_cpu_input_is_rejected_not_emulated():
    m = G.NeuralCAGraph(16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 16, 40, 40), fire_rate=1.0)
    with pytest.raises(RuntimeError):
        G.FixedSobelPerception(16)(torch.zeros(1, 16, 8, 8))


def test_rng_side_effects_with_stubbed_kernel(monkeypatch):
    """forward(): exactly one random.sample (also at message_gain 0), one torch.rand iff fire_rate < 1 (SURVEY 8b)."""
    calls = {}

    def stub(self, x, fire_rate, fire_u, *, chosen, message_gain, want_attn=False):
        calls["chosen"], calls["fire_u"], calls["gain"] = list(chosen), fire_u, message_gain
        return x
    monkeypatch.setattr(_base.FusedStepMixin, "_fused_step", stub)
    m = G.NeuralCAGraph(16, message_gain=0.0)
    x = torch.zeros(2, 16, 8, 8)
    random.seed(9); torch.manual_seed(9)
    m(x, fire_rate=0.5)
    after = (random.random(), float(torch.rand(1)))
    random.seed(9); torch.manual_seed(9)
    chosen = random.sample(m.graph.offsets, 8)
    fu = torch.rand(2, 1, 8, 8)
    assert (random.random(), float(torch.rand(1))) == after
    assert calls["chosen"] == chosen and torch.equal(calls["fire_u"], fu) and calls["gain"] == 0.0
    random.seed(9); torch.manual_seed(9)
    m(x, fire_rate=1.0)
    assert calls["fire_u"] is None
    random.seed(9); torch.manual_seed(9)
    random.sample(m.graph.offsets, 8)
    r1 = random.random()
    random.seed(9); m(x, fire_rate=1.0)
    assert random.random() == r1
    # classic: no python-RNG draw at all
    c = G.NeuralCA(16)
    random.seed(1); c(x, fire_rate=1.0); v = random.random()
    random.seed(1); assert random.random() == v


def test_schedule_draws_like_sequential_forward_calls():
    from graph_neural_cellular_automata_b200.rollout import make_schedule
    m = G.NeuralCAGraph(16, message_gain=0.25, graph_zero_padded_shift=False)
    random.seed(4)
    s = make_schedule(m, 2, 8, 8, 5, fire_rate=1.0, message_every=3, device="cpu")
    random.seed(4)
    ref = [random.sample(m.graph.offsets, 8) for _ in range(5)]
    assert s.offsets.shape == (5, 8, 2) and s.offsets.dtype == torch.int8
    assert s.offsets.tolist() == [[list(o) for o in st] for st in ref]
    assert s.message_gain.tolist() == pytest.approx([0.25, 0.0, 0.0, 0.25, 0.0])
    assert s.max_offset == 4 and s.total_updates == 10 and s.fire_u is None
    s2 = make_schedule(m, 3, 8, 8, 4, fire_rate=[0.5, 0.6, 0.7, 0.8], steps=[4, 1, 2], device="cpu", seed=5)
    assert s2.total_updates == 7 and s2.steps.tolist() == [4, 1, 2] and s2.philox_seed == 5


def test_pool_semantics():
    from graph_neural_cellular_automata_b200.training.pool import SamplePool
    from graph_neural_cellular_automata_b200.utils.nca_init import make_seed, trainer_seed
    torch.manual_seed(0)
    pool = SamplePool(10, lambda batch_size=1: trainer_seed(16, 8, batch_size), device="cpu")
    assert len(pool) == 10 and pool.pool.shape == (10, 16, 8, 8)
    random.seed(2)
    idx, batch = pool.sample(4)
    random.seed(2)
    assert idx == random.sample(range(10), 4)
    batch += 1.0                                                     # a copy: the pool is untouched
    assert float(pool.pool[idx[0], 0].abs().sum()) == 0.0
    pool.replace(idx, batch)
    assert torch.equal(pool.pool[idx[1]], batch[1])
    s = make_seed(16, 8, 2)
    assert float(s.sum()) == 26.0 and float(s[:, :3].abs().sum()) == 0.0


def test_native_offset_sampling_is_the_python_stream():
    """draw_offsets_array (C block replay of MT19937 outputs) == T x random.sample(graph.offsets, k), state included."""
    import random
    import graph_neural_cellular_automata_b200 as G
    from graph_neural_cellular_automata_b200.modules import graph_augmentation as GA
    m = G.NeuralCAGraph(16, update_hidden=128, img_size=40, graph_zero_padded_shift=False)
    assert GA._words_sample_ok(m.graph.offsets, len(m.graph.offsets), 8)      # the block replay draw_offsets_array uses
    for seed, T in ((0, 4), (7, 96), (123, 400)):
        random.seed(seed)
        ref = [random.sample(m.graph.offsets, 8) for _ in range(T)]
        after = random.getstate()
        random.seed(seed)
        arr = m.graph.draw_offsets_array(T)
        assert random.getstate() == after                       # the stream continues exactly where T forwards leave it
        assert [[tuple(int(v) for v in o) for o in st] for st in arr] == [[tuple(o) for o in st] for st in ref]


def test_words_sampler_reports_short_blocks_and_keeps_the_stream():
    """gnca_host_sample_offsets_words: a block of raw MT19937 outputs that is too short is refused (the python side
    retries with a longer one), a sufficient block reproduces random.sample and reports the words it consumed."""
    import ctypes as C
    import random
    import numpy as np
    from graph_neural_cellular_automata_b200 import _lib
    from graph_neural_cellular_automata_b200.modules.graph_augmentation import build_offsets
    lib = _lib.load()
    offsets = build_offsets(4)
    n, k, T = len(offsets), 8, 50
    table = np.ascontiguousarray(np.asarray(offsets, dtype=np.int8).reshape(n, 2))
    out = np.empty((T, k, 2), np.int8)
    used = C.c_int32(0)
    random.seed(99)
    state = random.getstate()
    m = 4 * T * k
    words = random.getrandbits(32 * m).to_bytes(4 * m, "little")
    # T * k draws need at least T * k words: a shorter block must be refused, not read past its end
    rc = lib.gnca_host_sample_offsets_words(words, T * k - 1, table.ctypes.data, n, k, T, out.ctypes.data, C.byref(used))
    assert rc == _lib.GNCA_ERR_UNSUPPORTED
    rc = lib.gnca_host_sample_offsets_words(words, m, table.ctypes.data, n, k, T, out.ctypes.data, C.byref(used))
    assert rc == 0 and T * k <= used.value <= m
    random.setstate(state)
    ref = [random.sample(offsets, k) for _ in range(T)]
    after = random.getstate()
    assert out.tolist() == [[list(o) for o in st] for st in ref]
    random.setstate(state)
    random.getrandbits(32 * used.value)              # skipping exactly `used` outputs lands on the reference's state
    assert random.getstate() == after


def test_history_allocation_is_quantised_in_steps():
    """rollout.py sizes the BPTT record buffer / dense history for T rounded up to 64 steps, so that rollouts of slightly
    different lengths reuse one cached block (a fresh 29 GB cudaMalloc per new maximum cost 70 ms in the long regime)."""
    from graph_neural_cellular_automata_b200.rollout import _round_up_steps, _QUANT_SLACK_BYTES
    assert [_round_up_steps(t) for t in (0, 1, 16, 17, 64, 65, 79, 80, 128, 390, 400)] == \
           [0, 1, 16, 64, 64, 128, 128, 128, 128, 448, 448]
    assert _QUANT_SLACK_BYTES >= 1 << 30
