"""``read_live``: the host side of the word beam's live read-out rows (include/nsd_b200.h, nsd_ctc_word_beam_live), no GPU."""
import numpy as np

from neural_speech_decoder_b200.ctc import LIVE_HEADER, read_live


def row(committed, first, top, words, cap):
    r = np.full(LIVE_HEADER + cap, -1, dtype=np.int32)
    r[:LIVE_HEADER] = committed, first, top, int(top - first > cap)
    r[LIVE_HEADER:LIVE_HEADER + len(words)] = words
    return r


def test_committed_then_tentative():
    # words 0..2 were handed out before; the top hypothesis has 7 words, the first 5 agreed on by every live one
    assert read_live(row(5, 3, 7, [13, 14, 15, 16], 6)) == ([13, 14], [15, 16], False)
    # nothing new: all tentative, or nothing at all
    assert read_live(row(3, 3, 5, [8, 9], 4)) == ([], [8, 9], False)
    assert read_live(row(3, 3, 3, [], 4)) == ([], [], False)


def test_narrow_row():
    # the tentative tail is cut at cap; committed words are never cut while they fit
    assert read_live(row(4, 2, 9, [1, 2, 3], 3)) == ([1, 2], [3], False)
    # more committed words than the row holds: the first cap now, the rest with the next read-out, no tentative words
    assert read_live(row(8, 2, 9, [1, 2, 3], 3)) == ([1, 2, 3], [], True)
    assert read_live(row(8, 5, 9, [4, 5, 6], 3)) == ([4, 5, 6], [], False)


def test_whole_buffer():
    buf = np.stack([row(1, 0, 2, [7, 8], 4), row(0, 0, 0, [], 4)])
    assert read_live(buf) == [([7], [8], False), ([], [], False)]
