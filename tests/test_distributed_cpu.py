"""world_size-2 gloo test of the N>1 host logic (no GPU): shard bookkeeping, the logging
all_gather in global env order, max-over-ranks timing, and that the reset RNG stream of a GLOBAL env
id does not depend on which rank owns it."""
import os
import socket
import numpy as np
import torch
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    from isaacgymenvs_b200 import distributed as D
    from oracle import tasks_np as T
    r, l, w = D.init("gloo")
    n = 8
    off = D.env_id_offset(r, n)
    per_env = torch.arange(n, dtype=torch.float32) + 100.0 * r
    allr = D.gather_returns(per_env)
    tmax = D.max_over_ranks([1.0 + r, 5.0 - r])
    D.barrier()
    # reset stream of global env 11 (owned by rank 1 as local env 3), drawn through the owner's offset
    owner, local = D.owner_of(11, n)
    u = T.reset_uniforms(42, D.env_id_offset(owner, n) + local, 0, 4) if owner == r else None
    q.put((r, off, allr.numpy().tolist(), tmax, None if u is None else u.tolist()))
    torch.distributed.destroy_process_group()


def test_two_rank_gloo():
    port = _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=120) for _ in ps)
    for p in ps:
        p.join(60)
        assert p.exitcode == 0
    (r0, off0, g0, t0, u0), (r1, off1, g1, t1, u1) = res
    assert (off0, off1) == (0, 8)
    expect = [float(i) for i in range(8)] + [100.0 + i for i in range(8)]
    assert g0 == expect and g1 == expect                      # global env order on every rank
    assert t0 == [2.0, 5.0] and t1 == [2.0, 5.0]              # max over ranks
    from oracle import tasks_np as T
    assert u0 is None and np.allclose(u1, T.reset_uniforms(42, 11, 0, 4))   # sharding-independent stream


def test_hand_resets_do_not_depend_on_the_sharding():
    """ShadowHand's reset_idx / reset_target_pose draw from a stream keyed by the GLOBAL env id (env_id_offset), so 16 envs
    stepped as one shard or as two shards of 8 come out identical (numpy restatement of the kernel's host contract)."""
    import os as _os
    from oracle import tasks_np as T
    from tests.hand_common import golden_case
    gold = np.load(_os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "golden", "shadow_hand.npz"))
    st, P, actions = golden_case(gold, "a")
    n = 16
    cut = lambda d, sl: {k: (v[sl].copy() if isinstance(v, np.ndarray) and v.shape[:1] == actions.shape[:1] else v) for k, v in d.items()}
    whole, Pw = cut(st, slice(0, n)), cut(P, slice(0, n))
    whole["reset"][:] = 1
    T.hand_pre_physics(whole, actions[:n], dict(Pw, env_id_offset=0))
    parts = []
    for r in range(2):
        sl = slice(8 * r, 8 * r + 8)
        s_, P_ = cut(st, sl), cut(P, sl)
        s_["reset"][:] = 1
        T.hand_pre_physics(s_, actions[sl], dict(P_, env_id_offset=8 * r))
        parts.append(s_)
    for k in ("root", "dof_pos", "dof_vel", "cur_targets", "goal_states"):
        assert np.array_equal(whole[k], np.concatenate([p[k] for p in parts], 0)), k


def test_hand_random_forces_do_not_depend_on_the_sharding():
    """The per-step force draws (shadow_hand.py:700-709) are keyed by (step, reset count, GLOBAL env id): one shard of 16 envs
    and two shards of 8 apply the same forces, with and without a reset in the step."""
    import os as _os
    from oracle import tasks_np as T
    from tests.hand_common import golden_case
    gold = np.load(_os.path.join(_os.path.dirname(_os.path.abspath(__file__)), "golden", "shadow_hand_force.npz"))
    st, P, actions = golden_case(gold, "f")
    n = 16
    cut = lambda d, sl: {k: (v[sl].copy() if isinstance(v, np.ndarray) and v.shape[:1] == (256,) else v) for k, v in d.items()}
    for step in range(2):
        whole, Pw = cut(st, slice(0, n)), cut(P, slice(0, n))
        whole["force_prob"][:] = 0.8
        if step == 1:
            whole["reset"][:] = 0; whole["reset_goal"][:] = 0
        T.hand_pre_physics(whole, actions[:n], dict(Pw, env_id_offset=0))
        parts = []
        for r in range(2):
            sl = slice(8 * r, 8 * r + 8)
            s_, P_ = cut(st, sl), cut(P, sl)
            s_["force_prob"][:] = 0.8
            if step == 1:
                s_["reset"][:] = 0; s_["reset_goal"][:] = 0
            T.hand_pre_physics(s_, actions[sl], dict(P_, env_id_offset=8 * r))
            parts.append(s_)
        for k in ("obj_force", "force_prob"):
            assert np.array_equal(whole[k], np.concatenate([p[k] for p in parts], 0)), (step, k)
        assert (np.abs(whole["obj_force"]).sum(1) > 0).sum() >= 8
        # a different global id draws a different force
        other = cut(st, slice(0, 8)); other["force_prob"][:] = 0.8
        if step == 1:
            other["reset"][:] = 0; other["reset_goal"][:] = 0
        T.hand_pre_physics(other, actions[:8], dict(cut(P, slice(0, 8)), env_id_offset=1000))
        assert not np.array_equal(other["obj_force"], whole["obj_force"][:8])
