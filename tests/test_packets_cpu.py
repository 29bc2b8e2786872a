"""Host side of stepping from UART packets: the batch layout concat_packets builds, and the sensor table's
num_doppler_bins field against include/mmw.h."""
import numpy as np

from mmwave_msc_b200 import _lib
from mmwave_msc_b200.batched import concat_packets
from oracle import tlv_oracle as tlv
from test_scene_sensors_cpu import _header_struct


def test_concat_packets_layout():
    a = tlv.encode_packet(3, np.ones((4, 5)), 9, 0.0626)
    b = tlv.encode_packet(4, np.zeros((0, 5)), 9, 0.0626)
    blob, off = concat_packets([a, None, b, None])
    assert blob.dtype == np.uint8 and off.dtype == np.int64
    np.testing.assert_array_equal(off, [0, len(a), len(a), len(a) + len(b), len(a) + len(b)])
    assert bytes(blob[off[0]:off[1]]) == a and bytes(blob[off[2]:off[3]]) == b
    blob, off = concat_packets([None, None])
    assert blob.size == 0 and off.tolist() == [0, 0, 0]
    blob, off = concat_packets([])
    assert blob.size == 0 and off.tolist() == [0]


def test_num_doppler_bins_field_matches_header():
    fields, size = _header_struct("mmw_scene_sensor")
    assert fields[-1] == ("num_doppler_bins", 36, 4) and size == 40
    assert _lib.SceneSensor.num_doppler_bins.offset == 36
    assert _lib.SCENE_SENSOR_DTYPE.fields["num_doppler_bins"] == (np.dtype("<i4"), 36)
    assert "reserved" not in _lib.SCENE_SENSOR_DTYPE.names
    assert _lib.KERNEL_NAMES[7] == "packets"
