"""TEST INFRASTRUCTURE — the generated six-player games of SIXPLAYER.md §6 (az_env6_play / az_env6_record / az_env6_samples) restated
on the C oracle: the checker of those calls.

Every slot plays its game id (first + slot) with the seat to move playing the scripted agent (script6.script_action) when its bit of
`script` is set and the uniform-random player (Oracle6Game.random_action) otherwise, with the real-move dice of (seed, game, ply).
A finished game is counted and re-dealt (new_game(seed, game, ply)) at the top of the next iteration, as az_env6_rollout does.  The
plies of the seats in `record_seats` are staged as (image before the ply, action); when a game has ended its staged samples become one
block of samples6.sample_record records with a one-hot policy target, by the end of the call.  A running game keeps its staged samples
for the next call."""
import numpy as np

from oracle import pyoracle as po
from oracle.samples6 import sample_record
from oracle.script6 import script_action


def one_hot(action):
    pi = np.zeros(po.MOVES, np.float32)
    pi[action] = 1.0
    return pi


class Generated6:
    """the slots `game_ids` (default first .. first + n - 1) of one env6 after reset(seed): play() mirrors one az_env6_play call"""

    def __init__(self, n, first, seed, rules=None, game_ids=None):
        self.seed, self.rules = seed, rules if rules is not None else po.default_rules()
        self.ids = list(game_ids) if game_ids is not None else [first + g for g in range(n)]
        self.games = [po.Oracle6Game(self.rules) for _ in self.ids]
        for o, gid in zip(self.games, self.ids):
            o.new_game(seed, gid, 0)
        self.ply = [0] * len(self.ids)
        self.staged = [[] for _ in self.ids]
        self.counters = dict(steps=0, games=0, draws=0, wins=[0] * 6)

    def _block(self, k, status):
        blob = np.stack([sample_record(img, one_hot(a), status) for img, a in self.staged[k]]).tobytes()
        self.staged[k] = []
        return blob

    def play(self, script, record_seats, n_plies):
        """n_plies plies of every slot; returns the record blocks (bytes, one per game) of the games that ended with staged samples"""
        blocks, c = [], self.counters
        for k, (o, gid) in enumerate(zip(self.games, self.ids)):
            ply = self.ply[k]
            for _ in range(n_plies):
                st = o.status()
                if st != -1:
                    c["games"] += 1
                    if st == -2:
                        c["draws"] += 1
                    else:
                        c["wins"][st] += 1
                    if self.staged[k]:
                        blocks.append(self._block(k, st))
                    o.new_game(self.seed, gid, ply)
                cur = o.s.cur
                a = script_action(o) if (script >> cur) & 1 else o.random_action(self.seed, gid, ply)
                if (record_seats >> cur) & 1:
                    self.staged[k].append((o.image(), a))
                assert o.move(a, self.seed, gid, ply) == 0
                ply += 1
            self.ply[k] = ply
            if self.staged[k] and o.status() != -1:
                blocks.append(self._block(k, o.status()))
        c["steps"] += len(self.games) * n_plies
        return blocks

    def images(self):
        return np.stack([o.image() for o in self.games])


def play(n, first, seed, script, record_seats, n_plies, rules=None):
    """one az_env6_play call of n_plies on a fresh env of n games: (images [n, 108], counters, record blocks)"""
    g = Generated6(n, first, seed, rules)
    blocks = g.play(script, record_seats, n_plies)
    return g.images(), g.counters, blocks
