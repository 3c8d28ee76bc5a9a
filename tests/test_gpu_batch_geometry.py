"""GPU: the batched State entry points at real launch geometry, lane by lane against the CPU oracle.

The lock-step parity suite steps every lane of a batch together from the initial state, mostly inside one thread block.
Here a batch holds lanes of every depth at once (initial, mid-game, chance, terminal), spans several blocks of the ILP
kernels and ends in a ragged warp, and every output lands between guard bytes, so that a kernel that reads the wrong
lane, writes the wrong row or writes past its range fails.  Each lane's expected values come from replaying its recorded
action history through the oracle; large batches (2^18 + lanes) are compared device against device, with a sample of
lanes replayed.
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import open_spiel_b200 as b2
from open_spiel_b200 import _lib
from oracle_lib import OracleGame
from parity import mask_words_to_lists

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# at least one variant per rule core, plus the edges of its layout
VARIANTS = [
    "tic_tac_toe",
    "connect_four",
    "connect_four(rows=7,columns=8,x_in_row=5)",     # 8 actions: no mask in the status byte
    "breakthrough",
    "breakthrough(rows=5,columns=4)",
    "hex(board_size=5)",
    "hex",
    "hex(board_size=4,swap=True)",
    "go(board_size=9)",
    "go(board_size=3,komi=0.5)",                     # positional superko decides many moves: history matters
    "kuhn_poker",
    "kuhn_poker(players=3)",
    "kuhn_poker(players=5)",
    "leduc_poker",
    "leduc_poker(players=3)",
    "leduc_poker(players=4)",
    "othello",
    "mnk",
    "mnk(m=15,n=15,k=3)",
    "y(board_size=11)",
    "havannah",
    "havannah(board_size=4,swap=True)",
]
# 2085 = 2 * (256 * 4) + 37: two full blocks at ILP <= 4 and a last warp with 5 live lanes
SIZES = [1, 33, 2085]
BIG = 2085
SPARE = 27            # batch capacity beyond n: lanes the calls with n lanes must not touch
GUARD = 256           # guard bytes on either side of every output
FILL = 0xA5           # guard / untouched-output byte


def _info_state(gs):
    return gs.startswith(("kuhn_poker", "leduc_poker"))


def _width(info):
    return max(info.num_distinct_actions, info.max_chance_outcomes)


def _compact_capable(info):
    return info.min_utility == -1.0 and info.max_utility == 1.0 and info.max_chance_outcomes == 0


class Guarded:
    """`rows` rows of `row_bytes` at byte `phase` past a 16-byte boundary, GUARD bytes of FILL before and after; every
    byte starts as FILL.  Device memory, or host memory (pinned or pageable)."""

    def __init__(self, rows, row_bytes, device, phase=0, pinned=False):
        self.lo, self.row_bytes = GUARD + phase, row_bytes
        t = torch.full((GUARD + phase + rows * row_bytes + GUARD,), FILL, dtype=torch.uint8, device=device)
        self.buf = t.pin_memory() if pinned else t
        assert self.buf.data_ptr() % 16 == 0

    @property
    def ptr(self):
        return self.buf.data_ptr() + self.lo

    def read(self, n, dtype, width=None):
        """Rows [0, n) as a numpy [n, width] array of `dtype`, after asserting that nothing else changed: the guards and
        the rows from n on still hold FILL."""
        h = self.buf.cpu().numpy() if self.buf.is_cuda else self.buf.numpy().copy()
        end = self.lo + n * self.row_bytes
        assert (h[:self.lo] == FILL).all(), "write before the output"
        assert (h[end:] == FILL).all(), "write past row n or past the output"
        v = h[self.lo:end].copy().view(dtype)
        return v.reshape(n, -1) if width is None else v.reshape(n, width)


def _stream(b):
    return b._stream()


def _ck(rc):
    _lib.check(rc)


# ---- mixed-depth batches -------------------------------------------------------------------------------------------

def _depth_bound(info):
    # max_game_length counts decisions only; the poker deals come on top, and this bound covers them
    return info.max_game_length * (2 if info.max_chance_outcomes > 0 else 1)


def build_mixed(game, n, seed, cap=None):
    """Batch of capacity `cap` whose lane i < n was advanced by its own uniform number of plies in [0, depth bound], each
    a uniformly chosen legal action (chance outcomes included) picked on the device; lanes >= n stay initial.  Returns the
    batch and the device action history [plies, n] (-1 once a lane has stopped)."""
    b = game.new_batch(cap or n)
    info, dev = b.info, b._dev
    g = torch.Generator(device=dev).manual_seed(seed)
    bound = _depth_bound(info)
    target = torch.randint(0, bound + 1, (n,), generator=g, device=dev)
    hist = torch.full((max(bound, 1), n), -1, dtype=torch.int32, device=dev)
    for ply in range(bound):
        a = random_legal(b, n, g)
        a = torch.where(target > ply, a, torch.full_like(a, -1))
        if not bool((a >= 0).any()):
            break
        hist[ply] = a
        b.apply_actions(a.contiguous(), n=n)
    assert b.error_count() == (0, -1)
    return b, hist


def random_legal(b, n, g):
    """One uniformly chosen legal action per lane, -1 on terminal lanes (device)."""
    acts, counts = b.legal_actions_list(n=n)
    idx = (torch.rand(n, generator=g, device=b._dev) * counts).long().clamp_(max=acts.shape[1] - 1)
    a = acts.gather(1, idx[:, None]).squeeze(1).to(torch.int32)
    return torch.where(counts > 0, a, torch.full_like(a, -1))


def replay(og, actions):
    st = og.new_initial_state()
    for a in actions:
        if a < 0:
            break
        st.apply_action(int(a))
    return st


def plies_of(actions):
    k = np.nonzero(np.asarray(actions) < 0)[0]
    return int(k[0]) if len(k) else len(actions)


class View:
    """Everything the read entry points report for a set of oracle states."""

    def __init__(self, states, P, info_state):
        self.cur = np.array([s.current_player() for s in states], dtype=np.int8)
        self.term = np.array([s.is_terminal() for s in states], dtype=np.uint8)
        self.rets = np.array([s.returns() for s in states], dtype=np.float32).reshape(len(states), P)
        self.legal = [s.legal_actions() for s in states]
        self.obs = np.stack([np.stack([s.observation_tensor(p) for s in states]) for p in range(P)])
        self.ist = np.stack([np.stack([s.information_state_tensor(p) for s in states]) for p in range(P)]) if info_state else None
        self.mover = np.maximum(self.cur.astype(np.int64), 0)


@functools.lru_cache(maxsize=None)
def mixed(gs, n):
    """(game, batch with capacity n + SPARE, host history [n, plies], oracle states, View); cached: tests only read it or
    copy from it."""
    game = b2.load_game(gs)
    b, hist = build_mixed(game, n, seed=n * 7919 + len(gs), cap=n + SPARE)
    hist = hist.t().cpu().numpy()
    og = OracleGame(gs)
    states = [replay(og, hist[i]) for i in range(n)]
    return game, b, hist, og, states, View(states, game.num_players(), _info_state(gs))


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def check_returns(got, want, what):
    # bit for bit, so the sign of a zero return counts
    np.testing.assert_array_equal(_bits(got), _bits(want), err_msg=what)


def check_mask(words, legal, width, what):
    got = mask_words_to_lists(torch.from_numpy(np.ascontiguousarray(words).view(np.int32)), width)
    for i, (g, w) in enumerate(zip(got, legal)):
        assert g == w, (what, i, g, w)


# ---- B: read entry points on a mixed-depth batch ---------------------------------------------------------------------

@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("gs", VARIANTS)
def test_read_entry_points_lane_by_lane(gs, n):
    game, b, hist, og, states, v = mixed(gs, n)
    info, dev, L = b.info, b._dev, _lib.lib()
    P, W, width, cap = info.num_players, info.mask_words, _width(info), b.n
    if n == BIG:     # the batch really mixes depths inside one warp
        kinds = np.where(v.term == 1, 0, np.where(v.cur == -1, 1, 2)).reshape(-1)[: n // 32 * 32].reshape(-1, 32)
        need = {0, 1, 2} if info.max_chance_outcomes > 0 else {0, 2}
        assert any(need <= set(row.tolist()) for row in kinds), "no warp mixes terminal, chance and decision lanes"
    for phase in range(4):
        cur, term = Guarded(cap, 1, dev, phase), Guarded(cap, 1, dev, phase)
        rets = Guarded(cap, 4 * P, dev, 4 * phase)
        _ck(L.b2s_status(b._h, cur.ptr, term.ptr, rets.ptr, n, _stream(b)))
        np.testing.assert_array_equal(cur.read(n, np.int8).reshape(-1), v.cur)
        np.testing.assert_array_equal(term.read(n, np.uint8).reshape(-1), v.term)
        check_returns(rets.read(n, np.float32, P), v.rets, gs + " returns")
    mask = Guarded(cap, 4 * W, dev)
    _ck(L.b2s_legal_mask(b._h, mask.ptr, n, _stream(b)))
    check_mask(mask.read(n, np.uint32, W), v.legal, width, gs + " mask")
    most = max(len(x) for x in v.legal)
    for stride in sorted({width, max(1, most // 2)}):
        acts, counts = Guarded(cap, 2 * stride, dev), Guarded(cap, 4, dev)
        _ck(L.b2s_legal_list(b._h, acts.ptr, counts.ptr, stride, n, _stream(b)))
        a, c = acts.read(n, np.int16, stride), counts.read(n, np.int32).reshape(-1)
        fill = np.full(1, FILL * 0x0101, dtype=np.uint16).view(np.int16)[0]
        for i, want in enumerate(v.legal):
            assert c[i] == len(want), (gs, "count", i)
            k = min(len(want), stride)
            assert a[i, :k].tolist() == want[:k], (gs, "legal list", i, stride)
            assert (a[i, k:] == fill).all(), (gs, "slot past the count", i, stride)
    tensors = [("obs", L.b2s_observation, info.observation_tensor_size, v.obs)]
    if v.ist is not None:
        tensors.append(("info", L.b2s_information_state, info.information_state_tensor_size, v.ist))
    for name, fn, F, want in tensors:
        for phase in range(4):
            for p in list(range(P)) + [-1]:
                out = Guarded(cap, 4 * F, dev, 4 * phase)
                _ck(fn(b._h, p, out.ptr, n, _stream(b)))
                got = out.read(n, np.float32, F)
                exp = want[p] if p >= 0 else want[v.mover, np.arange(n)]
                np.testing.assert_array_equal(got, exp, err_msg="%s %s player %d phase %d" % (gs, name, p, phase))


# ---- C: write entry points with a mixed action vector ------------------------------------------------------------------

def plant_actions(v, n, A, chance, seed):
    """Legal actions, -1 no-ops and illegal actions in one vector.  Lanes below 1024 (block 0 at ILP <= 4) get legal
    actions or -1; the bad lanes sit in blocks >= 1 and in the ragged tail.  Returns (actions, sorted bad lanes)."""
    rng = np.random.RandomState(seed)
    acts = np.full(n, -1, dtype=np.int32)
    for i in range(n):
        if not v.term[i] and rng.rand() < 0.75:
            acts[i] = v.legal[i][rng.randint(len(v.legal[i]))]
    lo = min(1024, n - 1)
    pool = list(rng.choice(np.arange(lo, n - 37), 10, replace=False)) + list(range(n - 37, n, 9))
    term = [i for i in range(lo, n) if v.term[i]]
    chn = [i for i in range(lo, n) if v.cur[i] == -1]
    pool += term[:1] + term[-1:] + chn[:2] + chn[-1:]
    bad = sorted(set(int(i) for i in pool))
    kinds = 0
    for i in bad:
        legal = set(v.legal[i])
        if v.term[i]:
            acts[i] = rng.randint(A)                       # any action on a terminal lane
        elif v.cur[i] == -1:
            out = [a for a in range(chance) if a not in legal]
            acts[i] = out[0] if out else chance            # a non-outcome at a chance node
        else:
            occupied = [a for a in range(A) if a not in legal]
            k = kinds % 3
            kinds += 1
            if k == 0 and occupied:
                acts[i] = occupied[rng.randint(len(occupied))]
            elif k == 1 or (k == 0 and not occupied):
                acts[i] = A + rng.randint(3)                # an id >= num_distinct_actions
            else:
                acts[i] = -2
    return acts, bad


def canon_blob(b, lane, plies):
    """The lane's packed state; for a history-keeping core only the history entries the state uses (0 .. ply)."""
    blob = b.state_blob(lane)
    if b.info.history_bytes:
        return blob[:b.info.state_bytes + 8 * (plies + 1)]
    return blob


def _status_byte(term, rets, mask_words, small):
    if term:
        return 0x80 | (1 if rets[0] > 0 else (2 if rets[0] < 0 else 0))
    return int(mask_words[0]) & 0x7F if small else 0


@pytest.mark.parametrize("gs", VARIANTS)
def test_write_entry_points_mixed_actions(gs):
    n = BIG
    game, snap, hist, og, states, v = mixed(gs, n)
    info, dev, L = snap.info, snap._dev, _lib.lib()
    P, W, A, width, cap = info.num_players, info.mask_words, info.num_distinct_actions, _width(info), snap.n
    acts, bad = plant_actions(v, n, A, info.max_chance_outcomes, seed=len(gs))
    # the oracle after the legal actions
    after = []
    plies = []
    for i, st in enumerate(states):
        p = plies_of(hist[i])
        if acts[i] >= 0 and i not in bad:
            st = st.clone()
            st.apply_action(int(acts[i]))
            p += 1
        after.append(st)
        plies.append(p)
    va = View(after, P, False)
    before = [canon_blob(snap, i, plies_of(hist[i])) for i in range(n)]
    work = game.new_batch(cap)
    a_d = torch.from_numpy(acts).to(dev)
    small = A <= 7

    def fresh():
        work.copy_from(snap, 0, 0, n)
        work._reset_errors()

    def finish(path):
        assert work.error_count() == (len(bad), bad[0]), (gs, path)
        blobs = [canon_blob(work, i, plies[i]) for i in range(n)]
        for i in bad:
            assert blobs[i] == before[i], (gs, path, "rejected lane changed", i)
        for i in range(n):
            if acts[i] == -1:
                assert blobs[i] == before[i], (gs, path, "no-op lane changed", i)
        return blobs

    def check_fused(path, mask, term, rets):
        if mask is not None:
            check_mask(mask, va.legal, width, (gs, path))
        if term is not None:
            np.testing.assert_array_equal(term.reshape(-1), va.term, err_msg=path)
        if rets is not None:
            check_returns(rets, va.rets, "%s %s returns" % (gs, path))

    results = {}
    # apply_actions: the other paths must leave the same states; this one is read back against the oracle
    fresh()
    work.apply_actions(a_d, n=n)
    results["apply"] = finish("apply")
    cur_, term_, rets_ = work.status(n=n)
    np.testing.assert_array_equal(cur_.cpu().numpy(), va.cur)
    check_fused("apply", work.legal_actions_mask_words(n=n).cpu().numpy().view(np.uint32), term_.cpu().numpy(),
                rets_.cpu().numpy())
    np.testing.assert_array_equal(work.observation_tensor(-1, n=n).cpu().numpy(), va.obs[va.mover, np.arange(n)])
    # fused step, device buffers
    fresh()
    mask, term, rets = Guarded(cap, 4 * W, dev), Guarded(cap, 1, dev), Guarded(cap, 4 * P, dev)
    _ck(L.b2s_step_fused(work._h, a_d.data_ptr(), mask.ptr, term.ptr, rets.ptr, n, _stream(work)))
    results["step"] = finish("step")
    check_fused("step", mask.read(n, np.uint32, W), term.read(n, np.uint8), rets.read(n, np.float32, P))
    # fused step, NULL outputs
    fresh()
    _ck(L.b2s_step_fused(work._h, a_d.data_ptr(), None, None, None, n, _stream(work)))
    results["step_null"] = finish("step_null")
    # host step, pinned and pageable
    for pinned in (True, False):
        fresh()
        a_h = Guarded(cap, 4, "cpu", pinned=pinned)
        a_h.buf[a_h.lo:a_h.lo + 4 * n].copy_(torch.from_numpy(acts.view(np.uint8)))
        mask, term, rets = (Guarded(cap, 4 * W, "cpu", pinned=pinned), Guarded(cap, 1, "cpu", pinned=pinned),
                            Guarded(cap, 4 * P, "cpu", pinned=pinned))
        _ck(L.b2s_step_fused_host(work._h, a_h.ptr, mask.ptr, term.ptr, rets.ptr, n))
        path = "step_host pinned=%s" % pinned
        results[path] = finish(path)
        check_fused(path, mask.read(n, np.uint32, W), term.read(n, np.uint8), rets.read(n, np.float32, P))
    # compact host step: uint8 (0xFF = no-op) and int32 actions, with and without the mask words
    if _compact_capable(info) and A <= 255:
        want = np.array([_status_byte(va.term[i], va.rets[i], [sum(1 << a for a in va.legal[i] if a < 32)], small)
                         for i in range(n)], dtype=np.uint8)
        for ab, dtype in ((1, np.uint8), (4, np.int32)):
            host_acts = np.where(acts == -1, 255, acts & 0xFF).astype(np.uint8) if ab == 1 else acts
            for with_mask in (False, True):
                fresh()
                a_h = Guarded(cap, ab, "cpu", pinned=True)
                a_h.buf[a_h.lo:a_h.lo + ab * n].copy_(torch.from_numpy(host_acts.astype(dtype).view(np.uint8)))
                status = Guarded(cap, 1, "cpu", pinned=True)
                mask = Guarded(cap, 4 * W, "cpu", pinned=True) if with_mask else None
                _ck(L.b2s_step_fused_host_compact(work._h, a_h.ptr, ab, status.ptr, mask.ptr if mask else None, n))
                path = "compact bytes=%d mask=%s" % (ab, with_mask)
                results[path] = finish(path)
                np.testing.assert_array_equal(status.read(n, np.uint8).reshape(-1), want, err_msg=path)
                if mask:
                    check_fused(path, mask.read(n, np.uint32, W), None, None)
    for path, blobs in results.items():
        assert blobs == results["apply"], (gs, path, "states differ from apply_actions")


# ---- D: host step at chunked and graph sizes -----------------------------------------------------------------------------

HOST_GAMES = ["tic_tac_toe", "connect_four", "breakthrough", "hex(board_size=5)", "go(board_size=9)", "kuhn_poker(players=3)",
              "kuhn_poker(players=5)", "leduc_poker", "leduc_poker(players=3)", "othello", "mnk(m=7,n=5,k=4)",
              "y(board_size=11)", "havannah(board_size=4)"]
HOST_N = (1 << 18) + 777
BAD_LANE = 135096          # in the second chunk for 2 and for 3 chunks


def _chunk_bounds(n, chunks):
    c = ((n + chunks - 1) // chunks + 1023) // 1024 * 1024       # enqueue_host_step's chunk length
    return list(range(c, n, c))


def _all_observables(b, n):
    cur, term, rets = b.status(n=n)
    return [cur, term, rets, b.legal_actions_mask_words(n=n), b.observation_tensor(-1, n=n)]


def host_step_check(gs, chunks, seed=3):
    """step_host with pinned buffers (graph path) and pageable buffers (stream path) against step on the device, over all
    lanes of a mixed-depth batch, plus a sample of lanes against the oracle."""
    n = HOST_N
    game = b2.load_game(gs)
    m, hist = build_mixed(game, n, seed)
    info, dev = m.info, m._dev
    P, W = info.num_players, info.mask_words
    x, y, z = game.new_batch(n), game.new_batch(n), game.new_batch(n)
    for t in (x, y, z):
        t.copy_from(m)
    g = torch.Generator(device=dev).manual_seed(seed + 1)
    a = random_legal(m, n, g)
    a = torch.where(torch.rand(n, generator=g, device=dev) < 0.25, torch.full_like(a, -1), a)
    a[BAD_LANE] = -2
    mz, tz, rz = z.step(a)
    outs = {}
    for t, pinned in ((x, True), (y, False)):
        a_h = Guarded(n, 4, "cpu", pinned=pinned)
        a_h.buf[a_h.lo:a_h.lo + 4 * n].copy_(a.cpu().view(torch.uint8))
        mask, term, rets = (Guarded(n, 4 * W, "cpu", pinned=pinned), Guarded(n, 1, "cpu", pinned=pinned),
                            Guarded(n, 4 * P, "cpu", pinned=pinned))
        _ck(_lib.lib().b2s_step_fused_host(t._h, a_h.ptr, mask.ptr, term.ptr, rets.ptr, n))
        outs[pinned] = (mask.read(n, np.uint32, W), term.read(n, np.uint8).reshape(-1), rets.read(n, np.float32, P))
    want = (mz.cpu().numpy().view(np.uint32), tz.cpu().numpy(), rz.cpu().numpy())
    for pinned, got in outs.items():
        for k in range(3):
            np.testing.assert_array_equal(got[k].view(np.uint8), want[k].view(np.uint8), err_msg="%s pinned=%s out %d" % (gs, pinned, k))
    for t in (x, y, z):
        assert t.error_count() == (1, BAD_LANE), gs
    oz = _all_observables(z, n)
    for t in (x, y):
        for u, w in zip(_all_observables(t, n), oz):
            assert torch.equal(u, w), gs
    # sampled lanes against the oracle: both sides of every chunk boundary and of several block boundaries
    rng = np.random.RandomState(seed)
    edges = _chunk_bounds(n, chunks) + [256, 512, 1024, 2048, 4096, 1 << 16, 1 << 17, 1 << 18]
    lanes = {0, n - 1, n - 2, BAD_LANE} | {e + d for e in edges for d in (-1, 0) if 0 <= e + d < n}
    lanes = sorted(lanes | set(rng.choice(n, 512 - len(lanes), replace=False).tolist()))
    idx = torch.tensor(lanes, device=dev)
    h = hist[:, idx].t().cpu().numpy()
    acts = a[idx].cpu().numpy()
    og = OracleGame(gs)
    states = []
    for j, lane in enumerate(lanes):
        st = replay(og, h[j])
        if acts[j] >= 0:
            st.apply_action(int(acts[j]))
        states.append(st)
    v = View(states, P, False)
    cur, term, rets, mask, obs = [o[idx].cpu().numpy() for o in oz]
    np.testing.assert_array_equal(cur, v.cur)
    np.testing.assert_array_equal(term, v.term)
    check_returns(rets, v.rets, gs)
    check_mask(mask.view(np.uint32), v.legal, _width(info), gs)
    np.testing.assert_array_equal(obs, v.obs[v.mover, np.arange(len(lanes))])


@pytest.mark.parametrize("gs", HOST_GAMES)
def test_host_step_chunked_and_graph_paths(gs):
    host_step_check(gs, chunks=2)


def test_host_step_three_chunks_in_a_fresh_process():
    """B2S_HOST_CHUNKS is read once per process: ragged multi-chunk views in a child process."""
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_batch_geometry as t\n"
            "for gs in ['go(board_size=9)', 'kuhn_poker(players=5)', 'hex(board_size=5)', 'leduc_poker(players=3)']:\n"
            "    t.host_step_check(gs, chunks=3)\nprint('ok')\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, B2S_HOST_CHUNKS="3")
    r = subprocess.run([sys.executable, "-c", code], env=env, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-3000:] + r.stderr[-3000:]


# the compact entry's games (win / loss / draw, no chance) with at most 255 actions, as uint8 actions need
ZC_GAMES = ["tic_tac_toe", "connect_four", "breakthrough(rows=5,columns=4)", "hex(board_size=5)", "go(board_size=9)", "othello",
            "mnk(m=7,n=5,k=4)", "y(board_size=11)", "havannah(board_size=4)"]


@pytest.mark.parametrize("gs", ZC_GAMES)
def test_zero_copy_step_ragged(gs):
    """Byte-wide host step with pinned, 16-byte aligned buffers: the kernel reads and writes host memory itself."""
    n = 6 * 1024 + 37
    game = b2.load_game(gs)
    m, _ = build_mixed(game, n, seed=9)
    info, dev = m.info, m._dev
    assert _compact_capable(info) and info.num_distinct_actions <= 255
    x, z = game.new_batch(n), game.new_batch(n)
    x.copy_from(m)
    z.copy_from(m)
    g = torch.Generator(device=dev).manual_seed(2)
    a = random_legal(m, n, g)
    a = torch.where(torch.rand(n, generator=g, device=dev) < 0.25, torch.full_like(a, -1), a)
    a[n - 3] = -2 & 0xFF           # uint8 254: out of range
    a[4100] = -2 & 0xFF
    mz, tz, rz = z.step(a)
    a_h = Guarded(n, 1, "cpu", pinned=True)
    a_h.buf[a_h.lo:a_h.lo + n].copy_(torch.where(a < 0, torch.full_like(a, 255), a).to(torch.uint8).cpu())
    status = Guarded(n, 1, "cpu", pinned=True)
    before = _lib.lib().b2s_host_zero_copy_steps()
    _ck(_lib.lib().b2s_step_fused_host_compact(x._h, a_h.ptr, 1, status.ptr, None, n))
    assert _lib.lib().b2s_host_zero_copy_steps() - before in (0, 1)     # 0 only where pinned memory is not device-mapped
    st = status.read(n, np.uint8).reshape(-1)
    tz, rz, mz = tz.cpu().numpy(), rz.cpu().numpy(), mz.cpu().numpy().view(np.uint32)
    small = info.num_distinct_actions <= 7
    want = np.array([_status_byte(tz[i], rz[i], mz[i], small) for i in range(n)], dtype=np.uint8)
    np.testing.assert_array_equal(st, want)
    assert x.error_count() == z.error_count() == (2, 4100)
    for u, w in zip(_all_observables(x, n), _all_observables(z, n)):
        assert torch.equal(u, w), gs


def test_host_graph_cache_eviction():
    """Five pinned buffer sets rotated on one batch, one more than the graphs it keeps: every call misses and evicts the
    least recently used graph, and every call must still equal the stream path."""
    gs, n = "go(board_size=9)", (1 << 16) + 333
    game = b2.load_game(gs)
    m, _ = build_mixed(game, n, seed=4)
    info, dev, L = m.info, m._dev, _lib.lib()
    P, W = info.num_players, info.mask_words
    x, y = game.new_batch(n), game.new_batch(n)
    x.copy_from(m)
    y.copy_from(m)
    sets = [[Guarded(n, k, "cpu", pinned=True) for k in (4, 4 * W, 1, 4 * P)] for _ in range(5)]
    g = torch.Generator(device=dev).manual_seed(8)
    graphs, calls = L.b2s_host_graph_launches(), 0
    for step in range(15):
        a = random_legal(y, n, g)
        acts_h, mask_h, term_h, rets_h = sets[step % 5]
        acts_h.buf[acts_h.lo:acts_h.lo + 4 * n].copy_(a.cpu().view(torch.uint8))
        _ck(L.b2s_step_fused_host(x._h, acts_h.ptr, mask_h.ptr, term_h.ptr, rets_h.ptr, n))
        calls += 1
        mu, tu, ru = torch.empty((n, W), dtype=torch.int32), torch.empty((n,), dtype=torch.uint8), torch.empty((n, P))
        y.step_host(a.cpu(), mu, tu, ru)
        assert np.array_equal(mask_h.read(n, np.uint32, W), mu.numpy().view(np.uint32)), step
        assert np.array_equal(term_h.read(n, np.uint8).reshape(-1), tu.numpy()), step
        assert np.array_equal(_bits(rets_h.read(n, np.float32, P)), _bits(ru.numpy())), step
    assert x.error_count() == y.error_count() == (0, -1)
    assert L.b2s_host_graph_launches() - graphs in (0, calls)   # 0 only where the capture is unsupported
    for u, w in zip(_all_observables(x, n), _all_observables(y, n)):
        assert torch.equal(u, w)


# ---- E: clones across capacities and offsets ------------------------------------------------------------------------------

CLONE_GAMES = ["tic_tac_toe", "connect_four", "breakthrough(rows=5,columns=4)", "hex(board_size=5)", "go(board_size=9)",
               "go(board_size=3,komi=0.5)", "kuhn_poker(players=3)", "leduc_poker", "leduc_poker(players=4)", "othello",
               "mnk(m=7,n=5,k=4)", "y(board_size=11)", "havannah(board_size=4,swap=True)"]


def play_out(b, lanes, ostates, gs, seed):
    """Plays lanes `lanes` of `b` to the end with random legal actions, in step with oracle states, comparing every
    observable at every ply; the other lanes get -1."""
    info, dev = b.info, b._dev
    P, width, info_state = info.num_players, _width(info), _info_state(gs)
    rng = np.random.RandomState(seed)
    idx = torch.tensor(lanes, device=dev)
    ply = 0
    while True:
        cur, term, rets = [t[idx].cpu().numpy() for t in b.status()]
        mask = b.legal_actions_mask_words()[idx].cpu()
        obs = [b.observation_tensor(p)[idx].cpu().numpy() for p in range(P)]
        ist = [b.information_state_tensor(p)[idx].cpu().numpy() for p in range(P)] if info_state else None
        v = View(ostates, P, info_state)
        np.testing.assert_array_equal(cur, v.cur, err_msg="%s ply %d" % (gs, ply))
        np.testing.assert_array_equal(term, v.term)
        check_returns(rets, v.rets, "%s ply %d" % (gs, ply))
        check_mask(mask.numpy().view(np.uint32), v.legal, width, (gs, ply))
        for p in range(P):
            np.testing.assert_array_equal(obs[p], v.obs[p], err_msg="%s ply %d player %d" % (gs, ply, p))
            if info_state:
                np.testing.assert_array_equal(ist[p], v.ist[p])
        acts = np.full(b.n, -1, dtype=np.int32)
        for j, lane in enumerate(lanes):
            if not v.term[j]:
                acts[lane] = v.legal[j][rng.randint(len(v.legal[j]))]
                ostates[j].apply_action(int(acts[lane]))
        if (acts < 0).all():
            break
        a = torch.from_numpy(acts).to(dev)
        if ply % 2:
            b.step(a)
        else:
            b.apply_actions(a)
        assert b.error_count() == (0, -1), (gs, ply)
        ply += 1


@pytest.mark.parametrize("gs", CLONE_GAMES)
def test_clones_across_capacities_and_offsets(gs):
    n = BIG
    game, src, hist, og, states, v = mixed(gs, n)
    dev, L = src._dev, _lib.lib()
    rng = np.random.RandomState(17)

    def oclone(lane):
        return states[lane].clone()

    # copy_from: smaller into larger, larger into smaller, with src_begin != dst_begin
    big = game.new_batch(src.n + 500)
    big.copy_from(src, src_begin=1700, dst_begin=2200, count=300)
    # broadcast_from into a sub-range: the deepest live lane
    live = [i for i in range(n) if not v.term[i]]
    deep = max(live, key=lambda i: plies_of(hist[i]))
    big.broadcast_from(src, deep, dst_begin=2530, count=40)
    small = game.new_batch(200)
    small.copy_from(src, src_begin=1234, dst_begin=37, count=150)
    # blob round trip into the small batch
    blob_pairs = [(190, 2060), (191, 5), (199, n - 1)]
    for d, s in blob_pairs:
        small.set_state_blob(d, src.state_blob(s))
        assert small.state_blob(d) == src.state_blob(s)
    # gather: repeated and permuted source lanes, one out-of-range index (checked: the destination lane is flagged)
    gat = game.new_batch(96)
    src_lanes = np.concatenate([rng.permutation(n)[:60], np.repeat([deep, n - 1], 18)])
    rng.shuffle(src_lanes)
    src_lanes = np.insert(src_lanes[:95], 61, src.n + 3).astype(np.int64)
    sl = torch.from_numpy(src_lanes).to(dev)
    gat._reset_errors()
    _ck(L.b2s_gather_states(gat._h, src._h, sl.data_ptr(), 96, _stream(gat)))
    assert gat.error_count() == (1, 61)
    gat._reset_errors()
    # play every clone to the end against an oracle clone of its source lane
    big_lanes = list(range(2200, 2500)) + list(range(2530, 2570))
    big_src = list(range(1700, 2000)) + [deep] * 40
    play_out(big, big_lanes, [oclone(s) for s in big_src], gs, 1)
    small_lanes = list(range(37, 187)) + [d for d, _ in blob_pairs]
    small_src = [oclone(s) for s in range(1234, 1384)] + [oclone(s) for _, s in blob_pairs]
    play_out(small, small_lanes, small_src, gs, 2)
    gat_src = [og.new_initial_state() if s >= src.n else oclone(int(s)) for s in src_lanes]
    play_out(gat, list(range(96)), gat_src, gs, 3)
    # the source batch is unchanged by all of it
    np.testing.assert_array_equal(src.status(n=n)[0].cpu().numpy(), v.cur)


def test_state_clone_and_child_on_go_follow_superko():
    gs = "go(board_size=3,komi=0.5)"
    game, og = b2.load_game(gs), OracleGame(gs)
    rng = np.random.RandomState(5)
    for trial in range(12):
        s, o = game.new_initial_state(), og.new_initial_state()
        for _ in range(rng.randint(4, 14)):
            if o.is_terminal():
                break
            a = rng.choice(o.legal_actions())
            s.apply_action(int(a))
            o.apply_action(int(a))
        if o.is_terminal():
            continue
        pairs = [(s.clone(), o.clone())]
        a = int(rng.choice(o.legal_actions()))
        oc = o.clone()
        oc.apply_action(a)
        pairs.append((s.child(a), oc))
        for ds, os_ in pairs:
            while True:
                assert ds.current_player() == os_.current_player()
                assert ds.legal_actions() == os_.legal_actions()
                check_returns(np.array(ds.returns()), np.array(os_.returns()), gs)
                for p in range(2):
                    np.testing.assert_array_equal(ds.observation_tensor(p), os_.observation_tensor(p))
                if os_.is_terminal():
                    assert ds.is_terminal()
                    break
                a = int(rng.choice(os_.legal_actions()))
                ds.apply_action(a)
                os_.apply_action(a)


# ---- F: returns buffers need 4-byte alignment only ------------------------------------------------------------------------

@pytest.mark.parametrize("gs", ["connect_four", "go(board_size=3,komi=0.5)", "kuhn_poker(players=3)"])
def test_returns_at_4_byte_offset(gs):
    game, b, hist, og, states, v = mixed(gs, BIG)
    info, dev, L = b.info, b._dev, _lib.lib()
    P, W, n = info.num_players, info.mask_words, BIG
    rets = Guarded(b.n, 4 * P, dev, phase=4)
    _ck(L.b2s_status(b._h, None, None, rets.ptr, n, _stream(b)))
    check_returns(rets.read(n, np.float32, P), b.status(n=n)[2].cpu().numpy(), gs)
    check_returns(rets.read(n, np.float32, P), v.rets, gs)
    x, y = game.new_batch(n), game.new_batch(n)
    x.copy_from(b, 0, 0, n)
    y.copy_from(b, 0, 0, n)
    a = random_legal(x, n, torch.Generator(device=dev).manual_seed(1))
    rets = Guarded(n, 4 * P, dev, phase=4)
    term = Guarded(n, 1, dev, phase=1)
    _ck(L.b2s_step_fused(x._h, a.data_ptr(), None, term.ptr, rets.ptr, n, _stream(x)))
    _, ty, ry = y.step(a)
    check_returns(rets.read(n, np.float32, P), ry.cpu().numpy(), gs)
    np.testing.assert_array_equal(term.read(n, np.uint8).reshape(-1), ty.cpu().numpy())
