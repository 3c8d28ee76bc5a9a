"""Pins the oracle restatement against the UNMODIFIED reference: random playouts, every observable after every move.
The reference's side is stored (tests/reference_golden.py): a digest of everything it showed along the same playouts."""
import zlib

import numpy as np
import pytest

from oracle_lib import OracleGame
from reference_golden import Digest, expected

GAMES = [
    ("tic_tac_toe", 60), ("connect_four", 60), ("connect_four(rows=4,columns=5,x_in_row=3)", 30),
    ("connect_four(rows=7,columns=8,x_in_row=5)", 30), ("connect_four(egocentric_obs_tensor=True)", 20),
    ("breakthrough", 30), ("breakthrough(rows=6,columns=6)", 20), ("breakthrough(rows=5,columns=4)", 20),
    ("hex", 25), ("hex(board_size=5)", 40), ("hex(num_cols=4,num_rows=3)", 40), ("hex(board_size=4,swap=True)", 40),
    ("hex(board_size=5,plain_obs_tensor=True)", 20), ("hex(num_cols=5,num_rows=3,plain_obs_tensor=True)", 20),
    ("go(board_size=9)", 25), ("go(board_size=5)", 60), ("go(board_size=7,komi=4.5)", 30),
    ("go(board_size=9,max_game_length=60)", 20), ("go(board_size=4,komi=0.5)", 80), ("go(board_size=3,komi=0.5)", 80),
    ("kuhn_poker", 100), ("kuhn_poker(players=3)", 100),
    ("havannah", 12), ("havannah(board_size=4)", 150), ("havannah(board_size=4,swap=True)", 150), ("havannah(board_size=6)", 40),
    ("havannah(board_size=2)", 100), ("havannah(board_size=3,swap=True)", 100), ("havannah(board_size=1)", 2),
    ("y(board_size=9)", 60), ("y(board_size=11)", 30), ("y(board_size=4)", 100), ("y(board_size=1)", 2), ("y", 5),
    ("othello", 60), ("mnk", 6), ("mnk(m=3,n=3,k=3)", 100), ("mnk(m=7,n=5,k=4)", 30), ("mnk(m=15,n=15,k=3)", 10), ("mnk(m=4,n=15,k=5)", 20),
    ("mnk(m=5,n=5,k=7)", 20), ("mnk(m=1,n=1,k=1)", 3),
    ("leduc_poker", 150), ("leduc_poker(players=3)", 80), ("leduc_poker(starting_player=1)", 50),
]


ATTRS = ("num_distinct_actions", "num_players", "max_game_length", "observation_tensor_size", "information_state_tensor_size",
         "max_chance_outcomes")


def observe(d, s):
    """Everything the comparison looks at in one state: returns with the sign of zero, tensors, strings, chance outcomes."""
    d.add(s.current_player(), s.is_terminal(), s.legal_actions(), [float(x).hex() for x in s.returns()], s.to_string())
    for p in range(s.game.num_players):
        d.add(s.observation_tensor(p))
        if s.game.information_state_tensor_size:
            d.add(s.information_state_tensor(p))
        d.add(s.information_state_string(p), s.observation_string(p))
    if s.is_chance_node():
        d.add(s.chance_outcomes())


def playouts(game, game_string, n_games):
    """Digest of n_games seeded random playouts; the moves are drawn from the implementation's own legal actions."""
    d = Digest([getattr(game, attr) for attr in ATTRS])
    rng = np.random.RandomState(zlib.crc32(game_string.encode()) % (2 ** 31))
    for _ in range(n_games):
        s = game.new_initial_state()
        while True:
            observe(d, s)
            if s.is_terminal():
                break
            la = s.legal_actions()
            s.apply_action(la[rng.randint(len(la))])
        d.add(s.history())
    return d.hexdigest()


def reference_golden():
    import ref_lib
    return {"ref_vs_oracle/" + gs: playouts(ref_lib.RefGame(gs), gs, n) for gs, n in GAMES}


@pytest.mark.parametrize("game_string,n_games", GAMES, ids=[g for g, _ in GAMES])
def test_oracle_equals_reference_on_random_playouts(game_string, n_games):
    assert playouts(OracleGame(game_string), game_string, n_games) == expected("ref_vs_oracle/" + game_string)
