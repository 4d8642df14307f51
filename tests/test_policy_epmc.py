"""Host restatement of the environmental-level policy (lifelike_agility_and_play_b200/policy_epmc.py; epmc_net.py:86-177): layer shapes of
the shipped files, TF 'SAME' convolutions against a brute-force evaluation, LSTM state handling.  The behavioural pin with the shipped
weights is tools/statistical_pin_epmc.py (DESIGN.md 6)."""
import numpy as np

from lifelike_agility_and_play_b200.policy_epmc import EpmcPolicy, _same_pad, conv1d_same_relu, conv2d_same_relu

from lifelike_agility_and_play_b200.policy_epmc import EPMC_SHAPES as SHAPES, SEPMC_SHAPES  # noqa: E402


def random_weights(seed=0):
    rng = np.random.default_rng(seed)
    w = [(rng.standard_normal(s) / np.sqrt(max(1, int(np.prod(s[:-1]))))).astype(np.float32) for s in SHAPES]
    w[1] = np.abs(w[1]) + 0.2
    return w


def test_shipped_layout_has_102_arrays():
    assert len(SHAPES) == 102


def test_same_convolutions_match_brute_force():
    rng = np.random.default_rng(3)
    for (H, W, k, s) in ((25, 13, 4, 2), (13, 7, 2, 2), (7, 4, 2, 1), (25, 13, 1, 1)):
        x = rng.standard_normal((2, H, W, 3)).astype(np.float32)
        w = rng.standard_normal((k, k, 3, 2)).astype(np.float32); b = rng.standard_normal(2).astype(np.float32)
        got = conv2d_same_relu(x, w, b, s)
        oh, pt, _ = _same_pad(H, k, s); ow, pl, _ = _same_pad(W, k, s)
        assert got.shape == (2, oh, ow, 2)
        ref = np.zeros_like(got)
        for n in range(2):
            for i in range(oh):
                for j in range(ow):
                    acc = b.copy()
                    for di in range(k):
                        for dj in range(k):
                            y, xx = i * s + di - pt, j * s + dj - pl
                            if 0 <= y < H and 0 <= xx < W:
                                acc = acc + x[n, y, xx] @ w[di, dj]
                    ref[n, i, j] = np.maximum(acc, 0)
        assert np.abs(got - ref).max() < 1e-4
    x = rng.standard_normal((2, 136, 1)).astype(np.float32)
    w = rng.standard_normal((4, 1, 4)).astype(np.float32)
    assert conv1d_same_relu(x, w, np.zeros(4, np.float32), 1).shape == (2, 136, 4)
    assert conv1d_same_relu(x[:, :128].repeat(4, 2), rng.standard_normal((4, 4, 4)).astype(np.float32), np.zeros(4, np.float32), 2).shape == (2, 64, 4)


def test_policy_structure_and_state():
    pol = EpmcPolicy(random_weights())
    rng = np.random.default_rng(1)
    obs = rng.standard_normal((6, 916)).astype(np.float32)
    s0 = pol.initial_state(6)
    a, s1, code = pol.act(obs, s0, np.ones(6, np.float32), return_code=True)
    assert a.shape == (6, 12) and s1.shape == (6, 64) and code.min() >= 0 and code.max() < 256 and np.isfinite(a).all()
    # the state matters, and the episode-start mask wipes it
    a2, s2 = pol.act(obs, s1, np.zeros(6, np.float32))
    a3, s3 = pol.act(obs, s1, np.ones(6, np.float32))
    assert not np.allclose(s2, s1) and np.allclose(s3, s1, atol=1e-6) and np.allclose(a3, a, atol=1e-6)
    # batch independence
    a4, s4 = pol.act(obs[2:3], s0[2:3], np.ones(1, np.float32))
    assert np.allclose(a4, a[2:3], atol=1e-5) and np.allclose(s4, s1[2:3], atol=1e-5)
    # only the proprioception is normalised and clipped
    big = obs.copy(); big[:, :135] = 1e6
    assert np.isfinite(pol.act(big, s0, np.ones(6, np.float32))[0]).all()


def test_strategic_policy_structure_and_state():
    from lifelike_agility_and_play_b200.policy_epmc import SepmcPolicy
    assert len(SEPMC_SHAPES) == 152
    rng = np.random.default_rng(5)
    w = [(rng.standard_normal(s) / np.sqrt(max(1, int(np.prod(s[:-1]))))).astype(np.float32) for s in SEPMC_SHAPES]
    w[1] = np.abs(w[1]) + 0.2
    pol = SepmcPolicy(w)
    obs = rng.standard_normal((4, 965)).astype(np.float32)
    s0 = pol.initial_state(4)
    a, s1, ang, code = pol.act(obs, s0, np.ones(4, np.float32), return_aux=True)
    assert a.shape == (4, 12) and s1.shape == (4, 128) and np.all(np.abs(ang) <= np.pi) and code.max() < 256 and np.isfinite(a).all()
    a2, s2 = pol.act(obs, s1, np.zeros(4, np.float32))
    a3, s3 = pol.act(obs, s1, np.ones(4, np.float32))
    assert not np.allclose(s2, s1) and np.allclose(s3, s1, atol=1e-6) and np.allclose(a3, a, atol=1e-6)
    # the game vector (opponent / flag) reaches the action only through the heading: the cheat copies of it (value tower inputs) do not
    o2 = obs.copy(); o2[:, 933:948] += 5.0; o2[:, 955:962] -= 3.0
    assert np.allclose(pol.act(o2, s0, np.ones(4, np.float32))[0], a, atol=1e-6)


import pytest  # noqa: E402


@pytest.mark.gpu
@pytest.mark.parametrize("strategic", [False, True])
def test_device_hierarchical_policy_matches_host(strategic):
    """csrc/llq_policy_hier.cu against the numpy statement of the same nets, random weights, three recurrent steps with episode starts in
    between: LSTM states to 1e-4, the same code for (almost) every row, actions to 1e-4 where the code agrees."""
    import torch
    from lifelike_agility_and_play_b200.policy_epmc import DeviceHierPolicy, SepmcPolicy
    rng = np.random.default_rng(11)
    shapes = SEPMC_SHAPES if strategic else SHAPES
    w = [(rng.standard_normal(s) / np.sqrt(max(1, int(np.prod(s[:-1]))))).astype(np.float32) for s in shapes]
    w[1] = np.abs(w[1]) + 0.2
    host = SepmcPolicy(w) if strategic else EpmcPolicy(w)
    dev = DeviceHierPolicy(w, device=0)
    n, ow, ld = 300, dev.obs_dim, dev.obs_dim + 7
    t_state = torch.zeros((n, dev.state_dim), device="cuda")
    t_act = torch.zeros((n, 12), device="cuda"); t_code = torch.zeros((n,), device="cuda", dtype=torch.int32)
    t_head = torch.zeros((n,), device="cuda")
    s_host = host.initial_state(n)
    same_total, rows = 0, 0
    for step in range(3):
        obs = np.zeros((n, ld), np.float32)
        obs[:, :ow] = rng.standard_normal((n, ow)).astype(np.float32)
        obs[:, 135:913] = np.abs(obs[:, 135:913]) * 0.7                 # distances / heights are non-negative in the env
        mask = (rng.uniform(size=n) < (1.0 if step == 0 else 0.3)).astype(np.float32)
        t_obs = torch.from_numpy(obs).cuda(); t_done = torch.from_numpy(mask.astype(np.uint8)).cuda()
        dev.forward(t_obs.data_ptr(), ld, n, t_done.data_ptr(), t_state.data_ptr(), t_act.data_ptr(), t_code.data_ptr(), t_head.data_ptr() if strategic else None)
        torch.cuda.synchronize()
        if strategic:
            a_ref, s_host, ang, c_ref = host.act(obs[:, :ow], s_host, mask, return_aux=True)
            assert np.abs(t_head.cpu().numpy() - ang).max() < 1e-4
        else:
            a_ref, s_host, c_ref = host.act(obs[:, :ow], s_host, mask, return_code=True)
        code = t_code.cpu().numpy(); same = code == c_ref
        same_total += int(same.sum()); rows += n
        st = t_state.cpu().numpy()
        assert np.abs(st - s_host).max() < 2e-4, np.abs(st - s_host).max()
        err = np.abs(t_act.cpu().numpy()[same] - a_ref[same]).max() / (1.0 + np.abs(a_ref).max())
        assert err < 1e-4, err
        s_host = st.copy()                                              # keep both sides on the same trajectory
    assert same_total >= 0.99 * rows, (same_total, rows)
    dev.close()


def test_role_table_points_at_arrays_of_the_right_shape():
    """include/llq_policy.h's roles -> arrays of the shipped files (policy_epmc.hier_role_arrays): a wrong index would still run."""
    from lifelike_agility_and_play_b200.policy_epmc import hier_role_arrays, _ENC, _LSTM, _LLC
    mlc = [(1, 135), (1, 135), (135, 64), (64,)] + _ENC + [(3, 32), (32,), (120, 64), (64,)] + [(128, 256), (256,)] + _LSTM + [(32, 256), (256,), (32, 256)] + _LLC[:10]
    hlc = [(135, 64), (64,)] + _ENC + [(88, 64), (64,)] + [(29, 64), (64,), (64, 64), (64,)] + [(192, 256), (256,)] + _LSTM + [(32, 1), (1,)]
    assert [SHAPES[i] for i in hier_role_arrays(False)] == mlc
    assert [SEPMC_SHAPES[i] for i in hier_role_arrays(True)] == mlc + hlc
    assert len(mlc) == 56 and len(mlc + hlc) == 101                      # LLQ_HIER_ROLES_MLC / LLQ_HIER_ROLES_ALL
