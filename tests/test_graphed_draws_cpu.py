"""The host half of train.HostDraws, the recorder through which GraphedStep stages the FPS start indices and the dropout
{seed, offset} of a train-mode forward, with a CPU control buffer (no GPU needed): the log, the re-staged values against the
eager draws, and the generator / dropout-counter state around recorded passes."""
import pytest
import torch

from pointnet12_b200 import train
from pointnet12_b200.model import pointnet_util
from pointnet12_b200.model.pointnet_util import draw_fps_starts
from pointnet12_b200.train import HostDraws, dropout_seed

# a mixed sequence of draw calls as a forward makes them: (B, level sizes) for FPS, None for a dropout
CALLS = [(4, (1024, 512)), None, (2, (64,)), None, (3, (2048, 512, 128))]
EXPECTED_LOG = [("fps", 4, (1024, 512)), ("dropout",), ("fps", 2, (64,)), ("dropout",), ("fps", 3, (2048, 512, 128))]
CTL_SIZE = 8 + 2 + 2 + 2 + 9


@pytest.fixture
def host_only(monkeypatch):
    """The eager draws stage through pinned memory; on a machine without a GPU the CPU tensor stands in for it."""
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self, *a, **k: self)
    monkeypatch.setitem(train._SEED, "next", 40)


def _forward():
    """The draw calls of CALLS, in order, as the nets make them -> what each returned."""
    out = []
    for c in CALLS:
        out.append(draw_fps_starts(c[0], list(c[1]), "cpu") if c is not None else dropout_seed("cpu"))
    return out


def _flat(values):
    return torch.cat([torch.stack(v).reshape(-1) if isinstance(v, list) else v for v in values])


def test_log_order_and_shapes(host_only):
    draws = HostDraws("cpu")
    with draws.recording():
        first = _forward()
    assert draws.log == EXPECTED_LOG
    assert draws.ctl.shape == (CTL_SIZE,) and draws.ctl.dtype == torch.int64
    assert [len(v) for v in first if isinstance(v, list)] == [2, 1, 3]
    with draws.recording():
        second = _forward()
    # the second pass hands out views of the control buffer, slice after slice in call order
    base = draws.ctl.data_ptr()
    o = 0
    for c, v in zip(CALLS, second):
        parts = v if isinstance(v, list) else [v]
        for t in parts:
            assert t.dtype == torch.int64 and t.shape == ((c[0],) if c is not None else (2,))
            assert t.data_ptr() == base + 8 * o
            o += t.numel()
    assert o == CTL_SIZE
    draws.ctl.copy_(torch.arange(CTL_SIZE))
    assert torch.equal(_flat(second), torch.arange(CTL_SIZE))
    assert pointnet_util.draw_log is None and train._SEED["next"] == 40


def test_a_pass_with_other_draws_is_refused(host_only):
    draws = HostDraws("cpu")
    with draws.recording():
        _forward()
    with pytest.raises(RuntimeError, match="HostDraws"):
        with draws.recording():
            dropout_seed("cpu")
    with pytest.raises(RuntimeError, match="HostDraws"):
        with draws.recording():
            _forward()
            dropout_seed("cpu")
    assert pointnet_util.draw_log is None


def test_restaged_values_equal_eager_draws(host_only):
    draws = HostDraws("cpu")
    with draws.recording():
        _forward()
    torch.manual_seed(1234)
    eager = [_flat(_forward()) for _ in range(3)]           # three eager iterations
    rng_eager, seed_eager = torch.get_rng_state(), train._SEED["next"]
    train._SEED["next"] = 40
    torch.manual_seed(1234)
    staged = []
    for _ in range(3):                                      # three replays
        buf = torch.zeros(CTL_SIZE, dtype=torch.int64)
        draws.draw_into(buf)
        staged.append(buf)
    for e, s in zip(eager, staged):
        assert torch.equal(e, s), (e, s)
    assert not torch.equal(staged[0], staged[1])            # every replay draws anew
    assert torch.equal(torch.get_rng_state(), rng_eager) and train._SEED["next"] == seed_eager == 46
    assert staged[2][8:10].tolist() == [torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, 45]


def test_recorded_passes_restore_generator_and_counter(host_only):
    torch.manual_seed(77)
    rng = torch.get_rng_state()
    draws = HostDraws("cpu")
    for _ in range(3):                                      # warm-up passes and the capture
        with draws.recording():
            _forward()
            torch.randint(0, 10, (5,))                      # anything else that consumes the generator inside the pass
            train._SEED["next"] += 3
    assert torch.equal(torch.get_rng_state(), rng) and train._SEED["next"] == 40
    with pytest.raises(ValueError):
        with draws.recording():
            torch.randint(0, 10, (5,))
            raise ValueError("a failing pass")
    assert torch.equal(torch.get_rng_state(), rng) and train._SEED["next"] == 40
    assert pointnet_util.draw_log is None
    # outside a recording the eager draws run as before
    v = dropout_seed("cpu")
    assert v.tolist() == [torch.initial_seed() & 0x7FFFFFFFFFFFFFFF, 41] and train._SEED["next"] == 41
    starts = draw_fps_starts(2, [100, 50], "cpu")
    assert not torch.equal(torch.get_rng_state(), rng) and [s.shape for s in starts] == [(2,), (2,)]
