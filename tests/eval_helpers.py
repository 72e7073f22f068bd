"""Host replays for evaluation-game tests: the Philox draw of the device opponent's default move
(csrc/selfplay.cu::philox_uniform53 with tag kTagOpponent) and a builder of packed game blocks
(the staged layout of include/mzb200.h)."""
import numpy

from oracle.philox import MASK, philox4x32_10

TAG_OPPONENT = 0x7169E005


def uniform53(seed, game, move, c2, tag):
    """csrc/selfplay.cu::philox_uniform53: counter (game lo, move, c2, game hi), key (seed lo, seed hi ^ tag), 53 bits."""
    x, y, _, _ = philox4x32_10((game & MASK, move & MASK, c2 & MASK, (game >> 32) & MASK),
                               (seed & MASK, ((seed >> 32) & MASK) ^ tag))
    return ((x >> 5) * 67108864.0 + (y >> 6)) * (1.0 / 9007199254740992.0)


def pack_block(game_id, slot, first_to_play, root_value, visits, action, reward, to_play, obs):
    """One staged game block (int64 game_id; int32 slot, T, first_to_play, O, A, bytes; then the arrays; pad to 8)."""
    visits = numpy.asarray(visits, numpy.int32)
    T, A = visits.shape
    obs = numpy.asarray(obs, numpy.float32).reshape(T + 1, -1)
    body = b"".join([numpy.asarray(root_value, numpy.float64).tobytes(), visits.tobytes(),
                     numpy.asarray(action, numpy.int32).tobytes(), numpy.asarray(reward, numpy.float32).tobytes(),
                     numpy.asarray(to_play, numpy.int32).tobytes(), numpy.zeros(T, numpy.float32).tobytes(), obs.tobytes()])
    size = (32 + len(body) + 7) & ~7
    head = numpy.array([game_id], numpy.int64).tobytes() + numpy.array(
        [slot, T, first_to_play, obs.shape[1], A, size], numpy.int32).tobytes()
    return (head + body).ljust(size, b"\0")
