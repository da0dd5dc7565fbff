"""GPU tests of the reference-facing Python surface: the drop-ins must behave like the classes
and functions they replace (TensorPoints, hironaka.src ops, hironaka/jax/util.py), written the
way the reference's own tests are (test/testTensorPoints.py, test/testJAX.py)."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from oracle import cport  # noqa: E402
from oracle import hk_oracle as O  # noqa: E402
from tests import kat as K  # noqa: E402

pytestmark = pytest.mark.gpu


def T(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def eq(t, a):
    return np.array_equal(t.detach().cpu().numpy(), np.asarray(a))


# ---- hironaka.src op surface (test/testTensorPoints.py:48-63) ---------------------------------
def test_src_functions():
    from hironaka_b200.src import (get_newton_polytope_torch, remove_repeated, reposition_torch, rescale_torch,
                                   shift_torch)
    p = T(K.R_IN)
    assert eq(get_newton_polytope_torch(p, inplace=False), K.R)
    assert eq(p, K.R_IN)  # inplace=False leaves the input alone
    assert get_newton_polytope_torch(p, inplace=True) is None
    assert eq(p, K.R)
    assert eq(shift_torch(p, [[1, 2], [0, 2, 3]], [1, 3], inplace=False), K.R2)
    shift_torch(p, [[1, 2], [0, 2, 3]], [1, 3], inplace=True)
    assert eq(p, K.R2)
    assert eq(reposition_torch(p, inplace=False), K.R3)
    reposition_torch(p, inplace=True)
    assert eq(p, K.R3)
    rescale_torch(p)
    assert eq(p, K.RS)
    q = T(K.REP_IN)
    remove_repeated(q)
    assert eq(q, K.REP_OUT)
    # multi-binary tensor form of coord and float axis (FusedGame passes both as float, fused_game.py:155)
    p = T(K.R)
    shift_torch(p, T(K.R_COORD_BIN), T(K.R_AXIS.astype(np.float32)))
    assert eq(p, K.R2)
    # non-contiguous input is still updated in place
    big = torch.zeros(2, 4, 8, device="cuda")
    view = big[:, :, :4]
    view.copy_(T(K.R_IN))
    get_newton_polytope_torch(view)
    assert eq(view, K.R)
    with pytest.raises(Exception):
        shift_torch(p, "bad", [1, 3])


# ---- TensorPoints (test/testTensorPoints.py:65-200) -------------------------------------------
def test_tensor_points_surface():
    from hironaka_b200 import TensorPoints
    pts = TensorPoints(T(K.R_IN))
    assert pts.batch_size == 2 and pts.max_num_points == 4 and pts.dimension == 4
    assert pts.get_newton_polytope() is pts and eq(pts.points, K.R)
    pts.shift([[1, 2], [0, 2, 3]], [1, 3])
    assert eq(pts.points, K.R2)
    pts.reposition()
    assert eq(pts.points, K.R3)
    pts.rescale()
    assert eq(pts.points, K.RS) and str(pts) == str(pts.points)

    pts = TensorPoints(T(K.R_IN))
    pts.get_newton_polytope()
    pts.shift([[1], [0, 2, 3]], [0, 1])
    assert eq(pts.points, K.R)  # both actions invalid: nothing happens
    pts = TensorPoints(T(K.ENDED_P)).copy()
    pts.shift([[0, 1]], [1], ignore_ended_games=True)
    assert eq(pts.points, K.ENDED_P)
    pts.shift([[0, 1]], [1], ignore_ended_games=False)
    assert eq(pts.points, K.ENDED_Q)

    p = TensorPoints(T(K.ORIGIN20_IN))
    p.get_newton_polytope()
    assert eq(p.points, K.ORIGIN20_OUT)
    assert p.ended and p.ended_batch_in_tensor.tolist() == [True] and p.get_num_points().tolist() == [1]

    point = TensorPoints(T(K.RESCALE0_IN))
    point.rescale()
    assert point.points.isfinite().all()

    a = TensorPoints(torch.rand(100, 20, 3))
    assert hash(a) == hash(a.copy()) and a.copy().points.data_ptr() != a.points.data_ptr()

    point = TensorPoints(T(K.RESCALE0_IN), dtype=torch.float32)
    point.type(torch.float16)
    assert point.dtype == torch.float16 and point.points.dtype == torch.float16

    # nested ragged list input with max_num_points (points_base / tensor_points.py:32-37)
    lst = [[[1, 2, 3], [2, 3, 4]], [[0, 1, 2]]]
    tp = TensorPoints(lst, max_num_points=3, padding_value=-1.0)
    assert eq(tp.points, [[[1, 2, 3], [2, 3, 4], [-1, -1, -1]], [[0, 1, 2], [-1, -1, -1], [-1, -1, -1]]])
    q = tp.get_newton_polytope(inplace=False)
    assert q is not tp and eq(tp.points[0, 1], [2, 3, 4]) and eq(q.points[0, 1], [-1, -1, -1])
    assert not tp.exceed_threshold()
    tp2 = TensorPoints(T(np.array([[[1e9, 0, 0], [0, 1, 0]]], np.float32)))
    assert tp2.exceed_threshold()
    from hironaka_b200 import HironakaB200Error
    with pytest.raises(HironakaB200Error):
        TensorPoints(torch.zeros(1, 2, 3), device="cpu")


def test_tensor_points_features_and_fused_game_flow():
    """The FusedGame.step composition (fused_game.py:54-102) against the oracle, with the
    experience filtering done the reference's way."""
    from hironaka_b200 import HostActionEncoder, TensorPoints
    rng = np.random.default_rng(3)
    B, N, d = 256, 20, 3
    x = rng.integers(0, 21, (B, N, d)).astype(np.float32)
    pts = TensorPoints(T(x))
    pts.get_newton_polytope()
    pts.rescale()
    ref = O.rescale_torch(O.get_newton_polytope_torch(x))
    assert eq(pts.points, ref)
    enc = HostActionEncoder(d)
    for t in range(5):
        obs = pts.get_features()
        done = pts.ended_batch_in_tensor
        assert eq(obs, O.get_features_torch(ref)) and eq(done, O.ended_batch(ref))
        hid = rng.integers(0, 4, B)
        host_move = enc.decode_tensor(T(hid))                   # [B, d] float multi-binary
        actions = host_move.argmax(1)                           # ChooseFirst agent
        pts.shift(host_move.type(pts.points.dtype), actions.type(pts.points.dtype))
        pts.get_newton_polytope()
        pts.rescale()
        ref = O.fused_game_point_ops(ref, host_move.cpu().numpy(), actions.cpu().numpy(), True)
        assert eq(pts.points, ref), t
        next_done = pts.ended_batch_in_tensor
        rew = next_done[~done].type(torch.float32)
        assert eq(rew, O.default_reward("host", O.ended_batch(ref))[~done.cpu().numpy()])


def test_list_points_order(golden_dir):
    """HK_F_OBS_SORT_LEX_FIRST and TensorPoints.to_list_points against the reference's ListPoints
    filter (tests/golden/ref_list_*.npz from get_newton_polytope_approx_lst)."""
    import glob, os
    from hironaka_b200 import TensorPoints, constants as C, ops
    for gen in (False, True):
        ops.force_generic(gen)
        for path in sorted(glob.glob(os.path.join(golden_dir, "ref_list_*.npz"))):
            g = np.load(path)
            for dt in (np.float32, np.int32):
                st = T(g["points"].astype(dt))
                r = ops.step(st, ops=C.HK_OP_NEWTON, flags=C.HK_F_OBS_SORT_LEX_FIRST, inplace=True, want_obs=True,
                             want_num_points=True)
                assert eq(r.obs.reshape(g["points"].shape), g["newton_list_order"]), (path, gen)
                assert eq(r.num_points, g["counts"])
            tp = TensorPoints(T(g["points"]))
            tp.get_newton_polytope()
            lst = tp.to_list_points()
            for b in range(len(lst)):
                assert lst[b] == g["newton_list_order"][b, : g["counts"][b]].tolist()
    ops.force_generic(False)


def test_fused_game_step_experiences():
    """hironaka_b200.FusedGame.step against the reference composition (fused_game.py:54-102):
    experiences of the games not already over, in order, with the pinned dtypes
    (test/testTrainer.py:105-118).  Deterministic players: a scripted host and ChooseFirst."""
    from hironaka_b200 import FusedGame, TensorPoints
    from hironaka_b200.players import AllCoordHostModule, ChooseFirstAgentModule, ChooseLastAgentModule

    class ScriptedHost(torch.nn.Module):
        def __init__(self, ids):
            super().__init__()
            self.ids, self.k = ids, 0

        def forward(self, x):
            out = torch.nn.functional.one_hot(self.ids[self.k % len(self.ids)].long(), num_classes=4).float()
            return out

    rng = np.random.default_rng(12)
    B, N, d = 300, 20, 3
    dev = torch.device("cuda")
    for sample_for, scale in (("host", True), ("agent", False)):
        x = rng.integers(0, 21, (B, N, d)).astype(np.float32)
        ids = [T(rng.integers(0, 4, B)) for _ in range(6)]
        host = ScriptedHost(ids)
        game = FusedGame(host, ChooseFirstAgentModule(d, N, dev), device=dev)
        pts = TensorPoints(T(x))
        pts.get_newton_polytope()
        ref = O.get_newton_polytope_torch(x)
        if scale:
            pts.rescale()
            ref = O.rescale_torch(ref)
        for t in range(5):
            host.k = t
            obs, act, rew, done, nobs = game.step(pts, sample_for, scale_observation=scale, exploration_rate=0.0)
            hid = ids[t].cpu().numpy()
            coords = O.decode_table(3)[hid].astype(np.float32)
            axis = coords.argmax(1)
            keep = ~O.ended_batch(ref)
            new = O.fused_game_point_ops(ref, coords, axis, scale)
            nd = O.ended_batch(new)
            assert rew.dtype == torch.float32 and done.dtype == torch.bool
            assert eq(done, nd[keep][:, None]) and eq(rew, O.default_reward(sample_for, nd[keep])[:, None])
            if sample_for == "host":
                assert act.dtype == torch.int32 and eq(act, hid[keep][:, None])
                assert eq(obs, O.get_features_torch(ref)[keep]) and eq(nobs, O.get_features_torch(new)[keep])
            else:
                assert eq(act, axis[keep][:, None]) and eq(obs["coords"], coords[keep])
                assert eq(obs["points"], O.get_features_torch(ref)[keep])
                assert eq(nobs["points"], O.get_features_torch(new)[keep])
            assert eq(pts.points, new)
            ref = new
    # the parameter-free players (test/testTrainer.py:36-46)
    ao = {"points": T(np.array([[[1, 0, 0]]], np.float32)), "coords": T(np.array([[1, 1, 0]], np.float32))}
    assert eq(ChooseFirstAgentModule(3, 20, dev)(ao), [[1.0, 0.0, 0.0]])
    assert eq(ChooseLastAgentModule(3, 20, dev)(ao), [[0.0, 1.0, 0.0]])
    assert eq(AllCoordHostModule(3, 20, dev)(ao["points"]), [[0.0, 0.0, 0.0, 1.0]])


def test_replay_buffer_masked_append_and_wraparound():
    """hk_experience_append: order-preserving compaction of the rows with skip == 0 into circular
    buffers with a device-resident position, against the reference procedure (boolean-mask filter
    then ReplayBuffer.add with wrap-around, replay_buffer.py:63-127) replayed in NumPy."""
    from hironaka_b200 import ReplayBuffer
    rng = np.random.default_rng(33)
    cap, N, d = 5000, 20, 3
    buf = ReplayBuffer({"points": (N, d), "coords": (d,)}, d, cap, torch.device("cuda"))
    ref = {k: np.zeros((cap,) + sh, np.float32) for k, sh in
           {"op": (N, d), "oc": (d,), "nop": (N, d), "noc": (d,)}.items()}
    ref_a, ref_r, ref_d = np.zeros((cap, 1), np.int32), np.zeros((cap, 1), np.float32), np.zeros((cap, 1), bool)
    pos, full = 0, False
    for it, B in enumerate([1, 31, 2048, 2049, 4999, 700, 3000]):
        skip = rng.random(B) < (0.5 if it % 2 else 0.1)
        op, nop = rng.random((B, N, d), dtype=np.float32), rng.random((B, N, d), dtype=np.float32)
        oc, noc = rng.integers(0, 2, (B, d)).astype(np.float32), rng.integers(0, 2, (B, d)).astype(np.float32)
        a, r, dn = rng.integers(0, 3, B).astype(np.int32), rng.random(B, dtype=np.float32), rng.random(B) < 0.3
        buf.add_masked(T(skip), {"points": T(op), "coords": T(oc)}, T(a), T(r), T(dn), {"points": T(nop), "coords": T(noc)})
        keep = ~skip
        L = int(keep.sum())
        for store, src in ((ref["op"], op), (ref["oc"], oc), (ref["nop"], nop), (ref["noc"], noc), (ref_a, a[:, None]),
                           (ref_r, r[:, None]), (ref_d, dn[:, None])):
            idx = (pos + np.arange(L)) % cap
            store[idx] = src[keep]
        full = full or (pos + L) >= cap
        pos = (pos + L) % cap
        assert buf.pos == pos and buf.full == full, it
    assert eq(buf.observations["points"], ref["op"]) and eq(buf.observations["coords"], ref["oc"])
    assert eq(buf.next_observations["points"], ref["nop"]) and eq(buf.next_observations["coords"], ref["noc"])
    assert eq(buf.actions, ref_a) and eq(buf.rewards, ref_r) and eq(buf.dones, ref_d)
    assert buf.actions.dtype == torch.int32 and buf.rewards.dtype == torch.float32 and buf.dones.dtype == torch.bool
    # the reference signature (already-filtered rows) and sampling
    buf2 = ReplayBuffer((N, d), 4, 100, torch.device("cuda"))
    o = torch.rand(7, N, d, device="cuda")
    buf2.add(o, torch.arange(7, device="cuda", dtype=torch.int32)[:, None], torch.ones(7, 1, device="cuda"),
             torch.zeros(7, 1, device="cuda", dtype=torch.bool), o + 1)
    assert buf2.pos == 7 and not buf2.full and torch.equal(buf2.observations[:7], o)
    so, sa, sr, sd, sn = buf2.sample(64)
    assert so.shape == (64, N, d) and int(sa.max()) <= 6 and torch.equal(sn, so + 1)


def test_fused_game_step_into_buffer_matches_step():
    """FusedGame.step_into (no host sync) fills the buffer with exactly what
    FusedGame.step + ReplayBuffer.add would."""
    from hironaka_b200 import FusedGame, ReplayBuffer, TensorPoints
    from hironaka_b200.players import AllCoordHostModule, ChooseLastAgentModule
    dev_ = torch.device("cuda")
    rng = np.random.default_rng(5)
    B, N, d = 500, 20, 3
    x = rng.integers(0, 21, (B, N, d)).astype(np.float32)
    for sample_for in ("host", "agent"):
        game = FusedGame(AllCoordHostModule(d, N, dev_), ChooseLastAgentModule(d, N, dev_), device=dev_)
        shape = (N, d) if sample_for == "host" else {"points": (N, d), "coords": (d,)}
        b1 = ReplayBuffer(shape, 4, 4096, dev_)
        b2 = ReplayBuffer(shape, 4, 4096, dev_)
        p1, p2 = TensorPoints(T(x)), TensorPoints(T(x))
        for p in (p1, p2):
            p.get_newton_polytope()
        for _ in range(4):
            b1.add(*game.step(p1, sample_for, scale_observation=False, exploration_rate=0.0))
            game.step_into(b2, p2, sample_for, scale_observation=False, exploration_rate=0.0)
        assert b1.pos == b2.pos and b1.pos > 0
        for a, b in ((b1.actions, b2.actions), (b1.rewards, b2.rewards), (b1.dones, b2.dones)):
            assert torch.equal(a, b)
        if sample_for == "host":
            assert torch.equal(b1.observations, b2.observations) and torch.equal(b1.next_observations, b2.next_observations)
        else:
            for k in ("points", "coords"):
                assert torch.equal(b1.observations[k], b2.observations[k])
                assert torch.equal(b1.next_observations[k], b2.next_observations[k])


def test_fused_game_graphed_step_into():
    """step_into captured in a CUDA graph: replays fill the buffer and move the points exactly as the
    eager calls do (deterministic players, no exploration), with the warm-up moves undone."""
    from hironaka_b200 import FusedGame, ReplayBuffer, TensorPoints
    from hironaka_b200.players import AllCoordHostModule, ChooseFirstAgentModule
    dev_ = torch.device("cuda")
    rng = np.random.default_rng(11)
    B, N, d = 4096, 5, 3
    x = -np.ones((B, N, d), np.float32)
    x[:, :4] = rng.integers(0, 9, (B, 4, d))
    for sample_for in ("host", "agent"):
        game = FusedGame(AllCoordHostModule(d, N, dev_), ChooseFirstAgentModule(d, N, dev_), device=dev_)
        shape = (N, d) if sample_for == "host" else {"points": (N, d), "coords": (d,)}
        b1, b2 = ReplayBuffer(shape, 4, 1 << 15, dev_), ReplayBuffer(shape, 4, 1 << 15, dev_)
        p1, p2 = TensorPoints(T(x)), TensorPoints(T(x))
        for p in (p1, p2):
            p.get_newton_polytope()
        graph = game.graphed_step_into(b2, p2, sample_for, scale_observation=True, exploration_rate=0.0)
        assert b2.pos == 0 and torch.equal(p1.points, p2.points)  # the warm-up left no trace
        for _ in range(5):
            game.step_into(b1, p1, sample_for, scale_observation=True, exploration_rate=0.0)
            graph.replay()
        torch.cuda.synchronize()
        assert b1.pos == b2.pos and b1.pos > 0
        assert torch.equal(p1.points, p2.points)
        n = b1.pos
        for a, b in ((b1.actions, b2.actions), (b1.rewards, b2.rewards), (b1.dones, b2.dones)):
            assert torch.equal(a[:n], b[:n])
        if sample_for == "host":
            assert torch.equal(b1.observations[:n], b2.observations[:n])
            assert torch.equal(b1.next_observations[:n], b2.next_observations[:n])
        else:
            for k in ("points", "coords"):
                assert torch.equal(b1.observations[k][:n], b2.observations[k][:n])
                assert torch.equal(b1.next_observations[k][:n], b2.next_observations[k][:n])


# ---- functional JAX-style API (test/testJAX.py:80-153,205-219,461-488) ------------------------
def test_functional_api():
    from hironaka_b200 import functional as F
    obs = torch.ones((32, 60), device="cuda")
    assert F.make_agent_obs(obs, torch.ones((32, 3), device="cuda")).shape == (32, 63)
    host_obs = T(K.TA_HOST_OBS)
    coords = T(K.TA_COORDS)
    ones = torch.ones(2, device="cuda")
    combined = torch.cat([host_obs.reshape(2, -1), coords], dim=1)
    ta = F.get_take_actions("host", (4, 3), rescale_points=True, reposition=False)
    out = ta(host_obs.reshape(2, -1), coords, ones)
    assert eq(out, O.take_actions("host", (4, 3), K.TA_HOST_OBS.reshape(2, -1), K.TA_COORDS, np.ones(2, np.float32), True, False))
    ta = F.get_take_actions("agent", (4, 3), rescale_points=False, reposition=False)
    out = ta(combined, ones, ones)
    assert eq(out, O.get_newton_polytope_jax(O.shift_jax(K.TA_HOST_OBS, K.TA_COORDS, np.ones(2))).reshape(2, -1))
    assert eq(host_obs, K.TA_HOST_OBS)  # functional: inputs untouched

    assert eq(F.get_feature_fn("host", (6, 3))(T(K.FEAT_IN.reshape(1, -1))), K.FEAT_SORTED)
    assert eq(F.get_feature_fn("agent", (3, 3), scale_observation=False)(T(K.AGENT_FEAT_IN)), K.AGENT_FEAT_NOSCALE)
    assert eq(F.get_feature_fn("agent", (3, 3), scale_observation=True)(T(K.AGENT_FEAT_IN)), K.AGENT_FEAT_SCALE)

    assert eq(F.get_dones(T(K.R)), [False, False]) and eq(F.get_dones(T(K.ORIGIN20_OUT)), [True])
    assert eq(F.get_done_from_flatten(T(K.AGENT_FEAT_IN), "agent", 3), [False, False])
    d, pd = torch.tensor([True, True, False]).cuda(), torch.tensor([False, True, False]).cuda()
    assert eq(F.get_reward_fn("host")(d, pd), [1, 0, 0]) and eq(F.get_reward_fn("agent")(d, pd), [-1, 0, 0])

    assert eq(F.decode_table(3), K.DECODE_3)
    assert eq(F.batch_encode(T(K.ENCODE_IN)), K.ENCODE_OUT)
    assert eq(F.batch_encode_one_hot(T(K.ENCODE_IN)), K.ENCODE_ONE_HOT_OUT)
    assert eq(F.get_batch_decode_from_one_hot(3)(T(K.ENCODE_ONE_HOT_OUT)), K.ENCODE_IN)
    assert eq(F.get_batch_decode(3)(T(K.ENCODE_OUT)), K.ENCODE_IN)
    with pytest.raises(ValueError):
        F.get_batch_decode(11)

    g = torch.Generator(device="cuda").manual_seed(0)
    pts = F.generate_pts(g, (64, 20, 3), 20, rescale=False, reposition=True)
    again = pts.clone()
    F.generate_pts  # root states are a fixed point of newton+reposition
    from hironaka_b200 import ops, constants as C
    ops.step(again, ops=C.HK_OP_NEWTON | C.HK_OP_REPOSITION, inplace=True)
    assert torch.equal(again, pts)


def test_value_targets_and_rollout_postprocess():
    """hk_value_targets vs the reference's vectors (test/testJAXTrainer.py:330-389) and vs the NumPy
    restatement on random rollouts.  Floating point: tolerance rtol 1e-5 / atol 1e-6 (the reference's
    own test uses jnp.isclose)."""
    from hironaka_b200 import functional as F
    for npts, role, unified, expect in K.VALUE_KATS:
        reward_role = "agent" if unified else role
        v = F.calculate_value_using_reward_fn(torch.zeros(npts.shape, device="cuda"), T(npts), 0.99, reward_role, role, unified)
        assert np.allclose(v.cpu().numpy(), expect, rtol=1e-5, atol=1e-6), (role, unified)
    pol, val = torch.zeros((1, 4, 3), device="cuda"), torch.zeros((1, 4), device="cuda")
    o, p_, v = F.rollout_postprocess((T(K.VALUE_OBS_AGENT), pol, val), "agent", 3, 0.99, True)
    assert np.allclose(v.cpu().numpy(), [-1, 1, -1, 1]) and o.shape == (4, 18) and p_.shape == (4, 3)
    v = F.rollout_postprocess((T(K.VALUE_OBS_HOST), pol, val), "host", 3, 0.99, True)[2]
    assert np.allclose(v.cpu().numpy(), [0.99, -1, 1, -1])
    rng = np.random.default_rng(2)
    for (B, Tn, N, d) in [(300, 20, 20, 3), (65, 7, 5, 3), (10, 40, 8, 4)]:
        # monotone point counts like a real game, then observations with that many live rows
        npts = np.sort(rng.integers(1, N + 1, (B, Tn)), axis=1)[:, ::-1].copy()
        for role in ("host", "agent"):
            for unified in (False, True):
                extra = d if (unified or role == "agent") else 0
                obs = -np.ones((B, Tn, N * d + extra), np.float32)
                for b in range(B):
                    for t in range(Tn):
                        obs[b, t, : npts[b, t] * d] = rng.random(npts[b, t] * d, dtype=np.float32)
                if extra:
                    obs[:, :, N * d:] = rng.integers(0, 2, (B, Tn, d))
                pol, val = np.zeros((B, Tn, 4), np.float32), np.zeros((B, Tn), np.float32)
                exp = O.rollout_postprocess(obs, pol, val, role, d, 0.97, unified)[2]
                got = F.rollout_postprocess((T(obs), T(pol), T(val)), role, d, 0.97, unified)[2].cpu().numpy()
                assert np.allclose(got, exp, rtol=1e-5, atol=1e-6), (B, Tn, role, unified)


def test_graphed_env_step():
    from hironaka_b200 import functional as F
    rng = np.random.default_rng(40)
    B, N, d = 100, 20, 3
    x = O.generate_pts(rng, (B, N, d), 20, rescale=False, reposition=True).astype(np.int32)
    for role in ("host", "agent"):
        g = F.GraphedEnvStep(role, (N, d), B)
        g.points.copy_(T(x))
        o = x
        for t in range(4):
            hid, ax, nxt = rng.integers(0, 4, B), rng.integers(0, 3, B), rng.integers(0, 4, B)
            g.host_action.copy_(T(hid.astype(np.int32)))
            g.axis.copy_(T(ax.astype(np.int32)))
            if role == "agent":
                g.next_coord.copy_(T(nxt.astype(np.int32)))
            pts, done, rew, obs = g()
            prev = O.get_dones(o.astype(np.float32))
            o, od, _, _ = cport.step(o, hid, ax, O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE)
            assert eq(pts, o) and eq(done, od.astype(bool)) and eq(rew, O.reward_fn(role, od.astype(bool), prev))
            exp_obs = cport.features(o, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE | O.F_ACT_DISCRETE,
                                     obs_coord=nxt.astype(np.int32) if role == "agent" else None)
            assert eq(obs, exp_obs)


def test_pack_coords_all_dtypes():
    from hironaka_b200.ops import coords_to_mask
    rng = np.random.default_rng(1)
    for d in (2, 3, 5, 10):
        mb = rng.integers(0, 2, (777, d))
        exp = (mb * (1 << np.arange(d))).sum(1).astype(np.int32)
        for dt in (torch.float32, torch.int32, torch.int64, torch.uint8, torch.bool, torch.float64, torch.float16):
            got = coords_to_mask(torch.as_tensor(mb).to(dt).cuda(), d, torch.device("cuda", 0))
            assert got.dtype == torch.int32 and eq(got, exp), (d, dt)


def test_fused_env_step_matches_composition():
    """get_env_step (one launch) == take_actions + get_dones + reward_fn + feature_fn."""
    from hironaka_b200 import functional as F
    rng = np.random.default_rng(9)
    B, N, d = 300, 20, 3
    x = O.generate_pts(rng, (B, N, d), 20, rescale=False, reposition=True)
    hid = rng.integers(0, 4, B)
    ax = rng.integers(0, 3, B)
    nxt = rng.integers(0, 4, B)
    coords = O.decode_table(3)[hid].astype(np.float32)
    for role in ("host", "agent"):
        env_step = F.get_env_step(role, (N, d), reposition=True, scale_observation=True)
        nx, done, rew, feat = env_step(T(x), T(hid.astype(np.int32)), T(ax.astype(np.int32)),
                                       next_coord=T(nxt.astype(np.int32)) if role == "agent" else None)
        exp = O.take_actions("host", (N, d), x.reshape(B, -1), coords, ax, False, True)
        assert eq(nx.reshape(B, -1), exp)
        exp_done = O.get_dones(exp.reshape(B, N, d))
        assert eq(done, exp_done) and eq(rew, O.reward_fn(role, exp_done, O.get_dones(x)))
        if role == "host":
            assert eq(feat, O.feature_fn("host", (N, d), exp, True))
        else:
            agent_obs = O.make_agent_obs(exp.reshape(B, N, d), O.decode_table(3)[nxt].astype(np.float32))
            assert eq(feat, O.feature_fn("agent", (N, d), agent_obs, True))


def test_game_batch_and_rho():
    from hironaka_b200 import GameBatch
    rng = np.random.default_rng(21)
    B, N, d, Tn = 4096, 20, 3, 12
    x = rng.integers(0, 20, (B, N, d)).astype(np.int32)
    ha = rng.integers(0, 4, (Tn, B)).astype(np.int32)
    ax = rng.integers(0, 3, (Tn, B)).astype(np.int32)
    gb = GameBatch(T(x), semantics="jax", reposition=True, initial_filter=True)
    gb2 = GameBatch(T(x), semantics="jax", reposition=True, initial_filter=True)
    o = cport.step(x, None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
    assert eq(gb.points, o)
    d0 = int(gb.dones().sum())
    counts = []
    for t in range(Tn):
        o, od, orw, _ = cport.step(o, ha[t], ax[t], O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE)
        done, rew = gb.step(T(ha[t]), T(ax[t]))
        assert eq(done, od.astype(bool)) and eq(rew, orw)
        counts.append(int(od.sum()))
    assert eq(gb.points, o)
    _, _, dcount, length = gb2.rollout(T(ha), T(ax))
    assert eq(gb2.points, o) and dcount.tolist() == counts
    rho = GameBatch.rho(d0, dcount, B)
    assert 0.0 < rho < 1.0
    assert eq(gb.features("host"), cport.features(o, O.F_OBS_SORT_LEX | O.F_OBS_RESCALE))


def test_compute_rho_matches_reference_loop():
    """engine.compute_rho (one launch per batch) against the reference's loop
    (jax_trainer.py:502-556) replayed with the oracle on the same root states, for fixed players."""
    from hironaka_b200 import compute_rho
    B, N, d, max_len, mv = 2000, 20, 3, 12, 20
    F = {"all_coord": 1 << 8, "zeillinger": 1 << 9, "choose_first": 1 << 10, "choose_last": 1 << 11}
    for host, agent in (("zeillinger", "choose_first"), ("all_coord", "choose_last"), ("zeillinger", "choose_last")):
        g = torch.Generator(device="cuda").manual_seed(7)
        rho, details = compute_rho(host, agent, B, (N, d), mv, max_len, num_of_loops=2, reposition=True, generator=g)
        g = torch.Generator(device="cuda").manual_seed(7)
        exp = [0] * max_len
        for _ in range(2):
            pts = torch.randint(0, mv, (B, N, d), generator=g, device="cuda", dtype=torch.int32).cpu().numpy()
            o = cport.step(pts, None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
            prev_done, done = 0, int(O.get_dones(o.astype(np.float32)).sum())
            for step in range(max_len - 1):
                exp[step] += done - prev_done
                o, od, _, _ = cport.step(o, None, None, O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, F[host] | F[agent])
                prev_done, done = done, int(od.sum())
            exp[max_len - 1] += B - done
        assert details == exp, (host, agent)
        assert abs(rho - sum(exp[1:]) / sum(i * v for i, v in enumerate(exp))) < 1e-12
    # random vs random: the players are drawn in the kernel (Philox keyed by seed << 20 | loop); the oracle replays
    # the documented streams
    g = torch.Generator(device="cuda").manual_seed(11)
    rho, details = compute_rho("random", "random", 4096, (20, 3), 20, 20, num_of_loops=2, generator=g, seed=5)
    g = torch.Generator(device="cuda").manual_seed(11)
    exp = [0] * 20
    for loop in range(2):
        pts = torch.randint(0, 20, (4096, 20, 3), generator=g, device="cuda", dtype=torch.int32).cpu().numpy()
        o = cport.step(pts, None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
        ha, ax = O.random_player_actions(4096, 3, 19, (5 << 20) + loop)
        prev_done, done = 0, int(O.get_dones(o.astype(np.float32)).sum())
        for step in range(19):
            exp[step] += done - prev_done
            o, od, _, _ = cport.step(o, ha[step], ax[step], O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON, O.F_ACT_DISCRETE)
            prev_done, done = done, int(od.sum())
        exp[19] += 4096 - done
    assert details == exp and 0 < rho < 1


def test_in_kernel_random_players():
    """HK_F_HOST_RANDOM / HK_F_AGENT_RANDOM (hk_rollout_seeded): the rollout with players drawn in the kernel equals
    the rollout fed with the documented Philox streams (oracle restatement, and hk_random_actions), in one launch
    or cut into calls with step_offset, on both kernel families, with one or both players random."""
    from hironaka_b200 import constants as C, ops
    rng = np.random.default_rng(31)
    op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    for (B, N, d) in [(5000, 20, 3), (700, 10, 3), (600, 64, 5), (300, 16, 4)]:
        Tn, seed = 9, 0x1234567890ABCDEF ^ B
        x = rng.integers(0, 15, (B, N, d)).astype(np.int32)
        ha, ax = O.random_player_actions(B, d, Tn, seed)
        gha, gax = ops.random_actions(B, d, Tn, seed)
        assert eq(gha, ha) and eq(gax, ax)
        assert ha.min() >= 0 and ha.max() == 2 ** d - d - 2 and ax.min() == 0 and ax.max() == d - 1
        o, counts = x, []
        for t in range(Tn):
            o, od, _, _ = cport.step(o, ha[t], ax[t], op_bits, O.F_ACT_DISCRETE)
            counts.append(int(od.sum()))
        out, _, _, dc, _ = ops.rollout_random(T(x), Tn, seed, ops=op_bits, flags=C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM,
                                              inplace=False)
        assert eq(out, o) and dc.tolist() == counts, (B, N, d)
        # cut into three calls: the step counter carries on
        st = T(x)
        got = []
        for (t0, n) in ((0, 4), (4, 1), (5, 4)):
            _, _, _, dc, _ = ops.rollout_random(st, n, seed, ops=op_bits, flags=C.HK_F_HOST_RANDOM | C.HK_F_AGENT_RANDOM,
                                                step_offset=t0)
            got += dc.tolist()
        assert eq(st, o) and got == counts, (B, N, d)
        # one player random, the other from a stream / fixed
        o2 = x
        ax_s = rng.integers(0, d, (Tn, B)).astype(np.int32)
        for t in range(Tn):
            o2 = cport.step(o2, ha[t], ax_s[t], op_bits, O.F_ACT_DISCRETE)[0]
        out2, *_ = ops.rollout_random(T(x), Tn, seed, ops=op_bits, flags=C.HK_F_HOST_RANDOM, axes=T(ax_s), inplace=False)
        assert eq(out2, o2), (B, N, d)
        o3 = x
        for t in range(Tn):
            o3 = cport.step(o3, None, ax[t], op_bits, 1 << 9)[0]  # Zeillinger host, random agent
        out3, *_ = ops.rollout_random(T(x), Tn, seed, ops=op_bits, flags=C.HK_F_HOST_ZEILLINGER | C.HK_F_AGENT_RANDOM,
                                      inplace=False)
        assert eq(out3, o3), (B, N, d)


def test_host_session_numpy_only():
    """hk_session_*: host (NumPy) buffers in and out, no torch tensors involved."""
    from hironaka_b200 import HostSession
    rng = np.random.default_rng(4)
    B, N, d = 5000, 20, 3
    x = rng.integers(0, 20, (B, N, d)).astype(np.int32)
    s = HostSession(x)
    ops_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    assert s.step(None, None, O.OP_NEWTON | O.OP_REPOSITION, 0) >= 0
    o = cport.step(x, None, None, O.OP_NEWTON | O.OP_REPOSITION, 0)[0]
    assert np.array_equal(s.get_state(), o)
    done = np.empty(B, np.uint8)
    rew = np.empty(B, np.float32)
    for t in range(4):
        ha, ax = rng.integers(0, 4, B).astype(np.int32), rng.integers(0, 3, B).astype(np.int32)
        cnt = s.step(ha, ax, ops_bits, O.F_ACT_DISCRETE, done=done, reward=rew)
        o, od, orw, _ = cport.step(o, ha, ax, ops_bits, O.F_ACT_DISCRETE)
        assert np.array_equal(done, od) and np.array_equal(rew, orw) and cnt == int(od.sum())
    assert np.array_equal(s.get_state(), o)
    s.close()


def test_uint8_actions_and_session_rollout():
    """HK_F_ACT_U8 (2 action bytes per game-step) and the pipelined host-buffer rollout."""
    from hironaka_b200 import HostSession, constants as C, ops
    rng = np.random.default_rng(17)
    for (B, N, d) in [(3000, 20, 3), (500, 64, 5)]:
        ncls = 2 ** d - d - 1
        Tn = 7
        x = rng.integers(0, 20, (B, N, d)).astype(np.int32)
        ha = rng.integers(0, ncls, (Tn, B)).astype(np.int32)
        ax = rng.integers(0, d, (Tn, B)).astype(np.int32)
        op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
        o, counts = x, []
        for t in range(Tn):
            o, od, _, _ = cport.step(o, ha[t], ax[t], op_bits, O.F_ACT_DISCRETE)
            counts.append(int(od.sum()))
        # device path with uint8 action tensors
        st = T(x)
        for t in range(Tn):
            hu, au = T(ha[t].astype(np.uint8)), T(ax[t].astype(np.uint8))
            rc_flags = C.HK_F_ACT_DISCRETE | C.HK_F_ACT_U8
            from hironaka_b200._lib import check, lib
            check(lib().hk_step(st.data_ptr(), st.data_ptr(), hu.data_ptr(), au.data_ptr(), None, None, None, None, None,
                                None, B, N, d, C.HK_DTYPE_I32, op_bits, rc_flags, -1.0, 1e8,
                                torch.cuda.current_stream().cuda_stream))
        assert eq(st, o)
        # one packed byte per game-step (HK_F_ACT_PACKED: id | axis << 5), per-step launches and a one-launch rollout
        packed = HostSession.pack_actions(ha, ax)
        st = T(x)
        for t in range(Tn):
            pk = T(packed[t])
            check(lib().hk_step(st.data_ptr(), st.data_ptr(), pk.data_ptr(), None, None, None, None, None, None, None,
                                B, N, d, C.HK_DTYPE_I32, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_PACKED, -1.0, 1e8,
                                torch.cuda.current_stream().cuda_stream))
        assert eq(st, o)
        st, pk = T(x), T(packed)
        dc = torch.zeros(Tn, dtype=torch.int32, device="cuda")
        check(lib().hk_rollout(st.data_ptr(), st.data_ptr(), pk.data_ptr(), None, None, None, dc.data_ptr(), None, B, N, d,
                               Tn, C.HK_DTYPE_I32, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_PACKED, -1.0,
                               torch.cuda.current_stream().cuda_stream))
        assert eq(st, o) and dc.tolist() == counts
        # packed actions are refused where they cannot be represented or make no sense
        assert lib().hk_step(st.data_ptr(), st.data_ptr(), pk.data_ptr(), None, None, None, None, None, None, None, B, N, d,
                             C.HK_DTYPE_I32, op_bits, C.HK_F_ACT_PACKED | C.HK_F_AGENT_FIRST, -1.0, 1e8,
                             torch.cuda.current_stream().cuda_stream) != 0
        # host-buffer session: int32, uint8 and packed streams
        for mode in ("i32", "u8", "packed"):
            s = HostSession(x)
            if mode == "packed":
                got = s.rollout(packed, None, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_PACKED)
            else:
                dt = np.uint8 if mode == "u8" else np.int32
                got = s.rollout(ha.astype(dt), ax.astype(dt), op_bits,
                                C.HK_F_ACT_DISCRETE | (C.HK_F_ACT_U8 if mode == "u8" else 0))
            assert got.tolist() == counts and np.array_equal(s.get_state(), o), mode
            s.close()
        # per-game done flags of every step read back on the third stream, several rollouts on one session
        # (the session's census carries over from call to call and is reset with the state)
        # The buffers are pinned and reused, so the second call captures the schedule as a CUDA graph and the
        # later ones replay it (the first runs eagerly).
        s = HostSession(x)
        oo = x
        packed_pin = torch.from_numpy(packed).pin_memory().numpy()
        done = torch.empty((Tn, B), dtype=torch.uint8).pin_memory().numpy()
        for rep in range(5):
            done[:] = 7
            got = s.rollout(packed_pin, None, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_PACKED, done=done)
            for t in range(Tn):
                oo, od, _, _ = cport.step(oo, ha[t], ax[t], op_bits, O.F_ACT_DISCRETE)
                assert np.array_equal(done[t], od), (rep, t)
                assert got[t] == int(od.sum()), (rep, t)
            assert np.array_equal(s.get_state(), oo), rep
            if rep == 2:  # a fresh state resets the census
                s.set_state(x)
                oo = x
        s.close()


def test_cuda_graph_capture_of_step():
    """The device entry points neither allocate nor synchronise: a step can be captured in a
    CUDA graph and replayed (MCTS node expansion, SURVEY.md section 7)."""
    from hironaka_b200 import ops, constants as C
    rng = np.random.default_rng(8)
    B, N, d = 512, 20, 3
    x = rng.integers(0, 20, (B, N, d)).astype(np.int32)
    state = T(x)
    ha = T(rng.integers(0, 4, B).astype(np.int32))
    ax = T(rng.integers(0, 3, B).astype(np.int32))
    op_bits = C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON
    ops.step(state, ha, ax, ops=op_bits, flags=C.HK_F_ACT_DISCRETE, inplace=True)  # warm up (smem opt-in)
    state.copy_(T(x))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        r = ops.step(state, ha, ax, ops=op_bits, flags=C.HK_F_ACT_DISCRETE, inplace=True, want_done=True)
    o = x
    for _ in range(3):
        g.replay()
        o = cport.step(o, ha.cpu().numpy(), ax.cpu().numpy(), op_bits, C.HK_F_ACT_DISCRETE)[0]
    torch.cuda.synchronize()
    assert eq(state, o) and eq(r.done, O.get_dones(o.astype(np.float32)))


def test_reference_arm_matches_the_gpu(golden_dir):
    """The unmodified reference (what `bench.py --impl reference` times) against the CUDA path the bench times
    (in-place census steps), bit for bit: states, done flags, rewards after every step.  The reference's torch
    ops treat an invalid action as a no-op and freeze ended games (hironaka/src/_torch_ops.py:90-93), so the
    kernel runs with those two flags here; the headline's JAX flavour is pinned by the JAX-source goldens.  The
    reference's side is stored: ref_rollout_c2_20x3*.npz, C2 random play recorded from the unmodified
    TensorPoints by oracle/gen_golden.py, tiled here to 4096 games.  Where baseline/_ref is installed, the live
    reference also plays the bench's own C2 inputs."""
    import os
    from baseline import reference_arm as R
    from hironaka_b200 import constants as C, ops
    flags = C.TORCH_SEMANTICS | C.HK_F_ACT_DISCRETE
    for name in ("c2_20x3", "c2_20x3_repos"):
        gd = np.load(os.path.join(golden_dir, f"ref_rollout_{name}.npz"))
        _, B, _, _, Tn, _, _, repos = gd["meta"].tolist()
        reps = -(-4096 // B)

        def tile(a):
            return np.tile(a, (reps,) + (1,) * (a.ndim - 1))
        step_ops = C.HK_OP_SHIFT | C.HK_OP_NEWTON | (C.HK_OP_REPOSITION if repos else 0)
        g = T(tile(gd["init"]).astype(np.int32))
        census = ops.new_census(g)
        ops.step(g, ops=C.HK_OP_NEWTON, inplace=True, census=census)
        assert np.array_equal(g.cpu().numpy().astype(np.float32), tile(gd["states"][0])), name
        for t in range(Tn):
            r = ops.step(g, T(tile(gd["host_ids"][t])), T(tile(gd["axes"][t])), ops=step_ops, flags=flags, inplace=True,
                         want_done=True, want_reward=True, census=census)
            assert np.array_equal(g.cpu().numpy().astype(np.float32), tile(gd["states"][t + 1])), (name, t)
            assert np.array_equal(r.done.cpu().numpy(), tile(gd["dones"][t + 1])), (name, t)
            assert np.array_equal(r.reward.cpu().numpy(),
                                  tile(gd["dones"][t + 1] & ~gd["dones"][t]).astype(np.float32)), (name, t)
    if not R.available():
        return
    import bench
    rtorch, TensorPoints, HostActionEncoder = R.import_reference()
    B, Tn = 4096, 20
    pts, ha, ax = bench.make_inputs(7, B, 1)
    tp = R.root_states(TensorPoints, rtorch, pts[0], True)
    rec = []
    R.play(tp, HostActionEncoder(3), rtorch, ha[0, :Tn], ax[0, :Tn], True, record=rec)
    g = T(pts[0])
    census = ops.new_census(g)
    root = C.HK_OP_NEWTON | C.HK_OP_REPOSITION
    ops.step(g, ops=root, inplace=True, census=census)
    flags = C.TORCH_SEMANTICS | C.HK_F_ACT_DISCRETE
    for t in range(Tn):
        r = ops.step(g, T(ha[0, t]), T(ax[0, t]), ops=C.HK_OP_SHIFT | C.HK_OP_REPOSITION | C.HK_OP_NEWTON, flags=flags,
                     inplace=True, want_done=True, want_reward=True, census=census)
        assert np.array_equal(g.cpu().numpy().astype(np.float32), rec[t][0]), t
        assert np.array_equal(r.done.cpu().numpy(), rec[t][1]) and np.array_equal(r.reward.cpu().numpy(), rec[t][2]), t


def test_done_bits_and_nibble_actions():
    """The compact transport of the end-to-end path: done flags as a bit mask (hk_step_census done_bits,
    hk_session_rollout_bits) and two games' actions per byte (HK_F_ACT_NIBBLE), both kernel families,
    ragged batch sizes, against the oracle on the unpacked actions."""
    from hironaka_b200 import HostSession, constants as C, ops
    rng = np.random.default_rng(23)
    op_bits = O.OP_SHIFT | O.OP_REPOSITION | O.OP_NEWTON
    for (B, N, d) in [(3001, 20, 3), (999, 10, 3), (64, 5, 3), (777, 33, 3)]:
        Tn = 9
        x = rng.integers(0, 12, (B, N, d)).astype(np.int32)
        x[::4, 2:] = -1
        ha = rng.integers(0, 4, (Tn, B)).astype(np.int32)
        ax = rng.integers(0, 3, (Tn, B)).astype(np.int32)
        nib = HostSession.pack_actions_nibble(ha, ax)
        assert nib.shape == (Tn, (B + 1) // 2)
        o = x
        g = T(x)
        census = ops.new_census(g)
        bits = torch.zeros((B + 31) // 32, dtype=torch.int32, device="cuda")
        ref_done = []
        for t in range(Tn):
            o, od, _, _ = cport.step(o, ha[t], ax[t], op_bits, O.F_ACT_DISCRETE)
            ref_done.append(od.astype(bool))
            bits.fill_(-1 if t % 2 else 0)  # every word must be written, whatever it held
            from hironaka_b200._lib import check, lib
            dn = torch.empty(B, dtype=torch.uint8, device="cuda")
            nb = T(nib[t])
            check(lib().hk_step_census(g.data_ptr(), nb.data_ptr(), None, dn.data_ptr(), bits.data_ptr(), None, None,
                                       census.data_ptr(), None, None, B, N, d, C.HK_DTYPE_I32, op_bits,
                                       C.HK_F_ACT_DISCRETE | C.HK_F_ACT_NIBBLE, -1.0, 1e8, torch.cuda.current_stream().cuda_stream))
            assert eq(g, o), (B, N, t)
            assert np.array_equal(dn.cpu().numpy().astype(bool), ref_done[-1]), (B, N, t)
            got = HostSession.unpack_done_bits(bits.cpu().numpy().view(np.uint32), B)
            assert np.array_equal(got, ref_done[-1]), (B, N, t)
        # host-buffer session: nibble stream up, bit masks down, graph replay from the second call on
        s = HostSession(x)
        nib_pin = torch.from_numpy(nib).pin_memory().numpy()
        bits_pin = torch.empty((Tn, (B + 31) // 32), dtype=torch.int32).pin_memory().numpy().view(np.uint32)
        for rep in range(3):
            s.set_state(x)
            bits_pin[:] = 0xdeadbeef
            counts = s.rollout(nib_pin, None, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_NIBBLE, done_bits=bits_pin)
            got = HostSession.unpack_done_bits(bits_pin, B)
            assert np.array_equal(got, np.stack(ref_done)), (B, N, rep)
            assert counts.tolist() == [int(r.sum()) for r in ref_done], (B, N, rep)
            assert np.array_equal(s.get_state(), o)
        s.close()
    # refused where it cannot be represented
    from hironaka_b200._lib import lib
    g = T(np.zeros((4, 16, 4), np.int32))
    assert lib().hk_step(g.data_ptr(), g.data_ptr(), g.data_ptr(), None, None, None, None, None, None, None, 4, 16, 4,
                         C.HK_DTYPE_I32, op_bits, C.HK_F_ACT_DISCRETE | C.HK_F_ACT_NIBBLE, -1.0, 1e8,
                         torch.cuda.current_stream().cuda_stream) != 0
