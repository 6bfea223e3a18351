"""build() decides whether libffb200.so is stale from one list of inputs: an edit to any source or header of
the library must rebuild it, or the tests would run the old kernels."""
import os

import __graft_entry__ as entry


def test_build_inputs_cover_every_source_and_header():
    inputs = entry.build_inputs()
    expected = {os.path.join(entry.CSRC, f) for f in os.listdir(entry.CSRC) if f.endswith(('.cu', '.cuh'))}
    expected.add(os.path.join(entry.ROOT, 'include', 'ffb200.h'))
    assert set(inputs) == expected
    for name in ('ffb_common.cuh', 'ffb_device.cuh', 'ffb_phase.cuh', 'ffb_peer.cuh', 'ffb_ctrlmat.cu'):
        assert os.path.join(entry.CSRC, name) in inputs
