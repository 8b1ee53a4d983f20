"""Host checks (no GPU) of the channel-count arguments: conv torsos take input_channels in [1, 16], and a
frame-deduplicated table takes [..., F] stacks and their flattened [..., C * F] form."""
import numpy as np
import pytest


@pytest.mark.parametrize('c', [0, 17, -1, 2.5, True])
def test_torso_rejects_channel_counts_outside_1_to_16(c):
  from acme_b200 import networks
  with pytest.raises(ValueError, match='input_channels'):
    networks.AtariTorso(input_channels=c)
  with pytest.raises(ValueError, match='input_channels'):
    networks.DQNAtariNetwork(4, input_channels=c)


def _table(shape, frame_stack, dtype=np.uint8):
  from acme_b200 import adders, replay, specs
  spec = specs.EnvironmentSpec(specs.Array(shape, dtype), specs.BoundedArray((6,), np.float32, -1., 1.),
                               specs.Array((), np.float32), specs.BoundedArray((), np.float32, 0., 1.))
  return replay.Table('t', replay.selectors.Uniform(), replay.selectors.Fifo(), max_size=10,
                      rate_limiter=replay.rate_limiters.MinSize(1), signature=adders.NStepTransitionAdder.signature(spec),
                      max_window=5, frame_stack=frame_stack)


@pytest.mark.parametrize('shape', [(84, 84, 4), (84, 84, 3, 4), (84, 84, 12), (84, 84, 1, 4)])
def test_frame_stack_accepts_stacks_and_flattened_stacks(shape):
  assert _table(shape, 4).frame_stack == 4


@pytest.mark.parametrize('shape,dtype', [((84, 84, 3), np.uint8), ((84, 84, 10), np.uint8), ((84, 84, 12), np.float32)])
def test_frame_stack_rejects_other_observations(shape, dtype):
  with pytest.raises(ValueError, match='frame_stack'):
    _table(shape, 4, dtype)
