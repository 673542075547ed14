"""TEST INFRASTRUCTURE — the six-player training record (include/az_b200.h AZ_SAMPLE6_BYTES) written on the host from its table, the
checker of az_selfplay6_samples and the input of the az_nn_train6 tests:

    bytes 0..107    the position before the move as its 108-byte r6_state image (Oracle6Game.image())
    bytes 108..111  float value target of the seat to move there: 1 when it won, 0 after a draw, -1/5 otherwise
    bytes 112..283  float policy target[43]
    byte  284       int8 final status (winner seat 0..5 or -2 = draw), bytes 285..287 zero
"""
import numpy as np

SAMPLE6_BYTES = 288
DRAW = -2
LOSS = np.float32(-1.0) / np.float32(5.0)     # the search's -v / 5 with v = 1, rounded to float like the device's __fdiv_rn


def sample_record(image, pi, status):
    """one record for the position `image` (108 bytes, seat to move = byte 98), policy target `pi` and final `status`"""
    img = np.ascontiguousarray(image, np.uint8).reshape(108)
    seat = int(img[98])
    value = np.float32(0.0) if status == DRAW else (np.float32(1.0) if status == seat else LOSS)
    out = np.zeros(SAMPLE6_BYTES, np.uint8)
    out[:108] = img
    out[108:112] = np.array([value], np.float32).view(np.uint8)
    out[112:284] = np.ascontiguousarray(pi, np.float32).reshape(43).view(np.uint8)
    out[284] = np.array([status], np.int8).view(np.uint8)[0]
    return out
