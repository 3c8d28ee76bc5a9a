"""Lock-step parity harness: CUDA batch (through the C ABI) vs the CPU oracle on the same seeded inputs.

Mirrors the reference's RandomSimTest (tests/basic_tests.cc:321-581): play random games to the end and check
every observable after every move — here with the oracle supplying the expected values.
"""
import numpy as np
import torch

import open_spiel_b200 as b2
from oracle_lib import OracleGame
from reference_golden import Digest


def mask_words_to_lists(words, width):
    """[n, W] int32 words -> list of ascending action lists."""
    w = words.cpu().numpy().astype(np.uint32)
    n = w.shape[0]
    bits = ((w[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(n, -1)[:, :width]
    return [np.nonzero(row)[0].tolist() for row in bits]


def lockstep(game_string, n_lanes=512, seed=0, check_obs_every=3, max_plies=None, check_info_state=False,
             checker=OracleGame):
    """Play n_lanes random games in lock-step on device and on the checker (the oracle restatement); assert equality of
    everything after every move.  checker=None: no checker; returns (steps, digest of everything a checker would have been
    compared with), to hold against checker_digest() of a checker that is not at hand (the unmodified reference)."""
    rng = np.random.RandomState(seed)
    game = b2.load_game(game_string)
    record = Digest(_header(game.num_distinct_actions(), game.max_game_length(), game.num_players(),
                            game.observation_tensor_size())) if checker is None else None
    if checker is not None:
        ogame = checker(game_string)
        assert game.num_distinct_actions() == ogame.num_distinct_actions
        assert game.max_game_length() == ogame.max_game_length
        assert game.num_players() == ogame.num_players
        assert game.observation_tensor_size() == ogame.observation_tensor_size
    batch = game.new_batch(n_lanes)
    ostates = [ogame.new_initial_state() for _ in range(n_lanes)] if checker is not None else [None] * n_lanes
    width = max(game.num_distinct_actions(), game.max_chance_outcomes())
    P = game.num_players()
    dev = batch._dev
    ply = 0
    total_steps = 0
    limit = max_plies or (game.max_game_length() + 8)
    while True:
        cur, term, rets = batch.status()
        cur, term, rets = cur.cpu().numpy(), term.cpu().numpy(), rets.cpu().numpy()
        legal = mask_words_to_lists(batch.legal_actions_mask_words(), width)
        acts_l, counts = batch.legal_actions_list()
        acts_l, counts = acts_l.cpu().numpy(), counts.cpu().numpy()
        obs = None
        if check_obs_every and ply % check_obs_every == 0:
            obs = [batch.observation_tensor(p).cpu().numpy() for p in range(P)]
            ist = [batch.information_state_tensor(p).cpu().numpy() for p in range(P)] if check_info_state else None
        actions = np.full(n_lanes, -1, dtype=np.int32)
        alive = 0
        for i, st in enumerate(ostates):
            if st is None:
                _record(record, cur[i], term[i], legal[i], rets[i].tolist(), obs and [o[i] for o in obs],
                        obs and check_info_state and [t[i] for t in ist])
                assert counts[i] == len(legal[i]) and acts_l[i, :len(legal[i])].tolist() == legal[i]
                if not term[i]:
                    actions[i] = legal[i][rng.randint(len(legal[i]))]
                    alive += 1
                continue
            assert int(cur[i]) == st.current_player(), (game_string, "current_player", i, ply)
            assert bool(term[i]) == st.is_terminal(), (game_string, "is_terminal", i, ply)
            ola = st.legal_actions()
            assert legal[i] == ola, (game_string, "legal", i, ply, legal[i], ola, st.to_string())
            assert counts[i] == len(ola) and acts_l[i, :len(ola)].tolist() == ola
            orets = st.returns()
            assert rets[i].tolist() == orets, (game_string, "returns", i, ply, rets[i], orets)
            assert np.array_equal(np.signbit(rets[i]), np.signbit(np.array(orets))), (game_string, "sign of zero")
            if obs is not None:
                for p in range(P):
                    np.testing.assert_array_equal(obs[p][i], st.observation_tensor(p),
                                                  err_msg="%s obs lane %d ply %d player %d\n%s" % (game_string, i, ply, p, st.to_string()))
                    if check_info_state:
                        np.testing.assert_array_equal(ist[p][i], st.information_state_tensor(p))
            if not st.is_terminal():
                a = ola[rng.randint(len(ola))]
                actions[i] = a
                st.apply_action(a)
                alive += 1
        if alive == 0:
            break
        total_steps += alive
        # alternate between the plain and the fused entry point
        a_d = torch.from_numpy(actions).to(dev)
        if ply % 2 == 0:
            batch.apply_actions(a_d)
        else:
            m, t, r = batch.step(a_d)
            # fused outputs must equal the separate calls made at the top of the next iteration
            cur2, term2, rets2 = batch.status()
            assert torch.equal(t, term2) and torch.equal(r, rets2)
            assert torch.equal(m, batch.legal_actions_mask_words())
        cnt, first = batch.error_count()
        assert cnt == 0, (game_string, "unexpected rejected lanes", cnt, first)
        ply += 1
        assert ply <= limit, "game did not end"
    return total_steps if record is None else (total_steps, record.hexdigest())


def _header(num_distinct_actions, max_game_length, num_players, observation_tensor_size):
    return [num_distinct_actions, max_game_length, num_players, observation_tensor_size]


def _record(d, cur, term, legal, rets, obs, ist):
    d.add(int(cur), bool(term), legal, [float(x).hex() for x in rets], obs or None, ist or None)


def checker_digest(game_string, checker, n_lanes=512, seed=0, check_obs_every=3, max_plies=None, check_info_state=False):
    """The checker's side of lockstep(checker=None): its states played the same way, observed the same way."""
    rng = np.random.RandomState(seed)
    g = checker(game_string)
    d = Digest(_header(g.num_distinct_actions, g.max_game_length, g.num_players, g.observation_tensor_size))
    states = [g.new_initial_state() for _ in range(n_lanes)]
    P = g.num_players
    ply = 0
    while True:
        check = check_obs_every and ply % check_obs_every == 0
        actions = []
        for st in states:
            la = st.legal_actions()
            _record(d, st.current_player(), st.is_terminal(), la, st.returns(),
                    check and [st.observation_tensor(p) for p in range(P)],
                    check and check_info_state and [st.information_state_tensor(p) for p in range(P)])
            actions.append(None if st.is_terminal() else la[rng.randint(len(la))])
        if all(a is None for a in actions):
            return d.hexdigest()
        for st, a in zip(states, actions):
            if a is not None:
                st.apply_action(a)
        ply += 1
