"""CPU suite: the six-player training record (AZ_SAMPLE6_BYTES = 288) as the test side writes it (oracle/samples6.py): the image before
the move, the six-seat value target, the policy target, the final status byte and zero padding; the size agrees with the C header and
the Python binding."""
import os
import re

import numpy as np

from oracle import pyoracle as po
from oracle import samples6

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SEED = 0x5EED0001


def test_record_size_agrees_with_header_and_binding():
    text = open(os.path.join(ROOT, "include", "az_b200.h")).read()
    assert int(re.search(r"#define AZ_SAMPLE6_BYTES (\d+)", text).group(1)) == samples6.SAMPLE6_BYTES == 288
    from alphazero_risk_b200 import api
    assert api.SAMPLE6_BYTES == samples6.SAMPLE6_BYTES


def test_sample_record_layout():
    rules = po.default_rules()
    o = po.Oracle6Game(rules)
    o.new_game(SEED, 17, 0)
    for ply in range(500):
        assert o.move(o.random_action(SEED, 17, ply), SEED, 17, ply) == 0
    assert o.status() == -1
    img, cur = o.image(), int(o.s.cur)
    assert img[98] == cur
    valid = o.valid()
    pi = np.array([(i + 1.0) if (valid >> i) & 1 else 0.0 for i in range(43)], np.float32)
    pi /= pi.sum()
    loser = (cur + 1) % 6
    for status, value in ((cur, np.float32(1.0)), (loser, np.float32(-1.0) / np.float32(5.0)), (-2, np.float32(0.0))):
        rec = samples6.sample_record(o.image(), pi, status)
        assert rec.dtype == np.uint8 and rec.shape == (samples6.SAMPLE6_BYTES,) == (288,)
        assert (rec[:108] == img).all()
        assert rec[108:112].view(np.float32)[0].view(np.uint32) == value.view(np.uint32)
        assert (rec[112:284].view(np.uint32) == pi.view(np.uint32)).all()
        assert rec[284:285].view(np.int8)[0] == status
        assert (rec[285:] == 0).all()
    assert (o.image() == img).all()
    # over the six possible winners the seat to move gets 1 once and -1/5 five times
    vals = [samples6.sample_record(img, pi, w)[108:112].view(np.float32)[0] for w in range(6)]
    assert sorted(vals)[-1] == 1.0 and vals.count(np.float32(-0.2)) == 5
