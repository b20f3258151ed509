"""Every route the results of a step with host buffers can take (te_api.cu: pick_route) gives, bit for bit, what the
same step gives on a handle stepped with device buffers: wire records expanded by the handle's threads, float arrays
written by the copy engine (TE_HOST_FLOAT_DMA=1), steps too long for a record (k_ticks > 13), masked steps, and the
records themselves - launched in one slice or in several (TE_HOST_SLICES)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

E, I, SEED = 301, 9, 17
KW = dict(m=3, n=3, length=250.0, num_envs=E, arrivals="philox", seed=SEED, local_cars_per_sec=0.6, ticks_per_step=10,
          remi=True)


def make_env(float_dma, slices):
    """A handle created under the given host-path switches (read once, at te_create)."""
    from traffic_env_b200 import VecTrafficEnv
    keys = ("TE_HOST_FLOAT_DMA", "TE_HOST_SLICES", "TE_HOST_THREADS")
    saved = {k: os.environ.get(k) for k in keys}
    os.environ.update(TE_HOST_FLOAT_DMA=str(float_dma), TE_HOST_SLICES=str(slices), TE_HOST_THREADS="2")
    try:
        return VecTrafficEnv(**KW)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("slices", [1, 3])
@pytest.mark.parametrize("float_dma", [0, 1])
def test_host_routes_equal_device_buffers(float_dma, slices):
    import torch
    from traffic_env_b200._lib import TE_CTRL_GREEDY, TE_DEVICE, check
    h = make_env(float_dma, slices)
    d = make_env(float_dma, slices)
    assert h.host_float_dma() == bool(float_dma)
    dev = torch.device("cuda", 0)
    OL, stride, done_at = h.obs_len, h.wire.stride, h.wire.done
    d_act = torch.zeros((2, E, I), dtype=torch.uint8, device=dev)
    d_obs = torch.zeros((3, E, OL), dtype=torch.float32, device=dev)
    d_rew = torch.zeros((3, E, I), dtype=torch.float32, device=dev)
    d_done = torch.zeros((3, E), dtype=torch.uint8, device=dev)
    d_rec = torch.zeros((3, E, stride), dtype=torch.uint8, device=dev)
    rng = np.random.RandomState(SEED)
    init = rng.randint(2, size=(E, I))
    h.reset(init_phase=init)
    d.reset(init_phase=init)

    def device_out(n):
        d.synchronize()
        return d_obs[:n].cpu().numpy(), d_rew[:n].cpu().numpy(), d_done[:n].cpu().numpy()

    def same(got, want, what):
        for g, w, name in zip(got, want, ("obs", "reward", "done")):
            assert np.ascontiguousarray(g).tobytes() == np.ascontiguousarray(w).tobytes(), (what, name)

    for rnd in range(3):
        tag = "round %d" % rnd
        for k in (10, 20):                     # 20 ticks: too long for a record, the float staging route
            act = rng.randint(2, size=(E, I)).astype(np.uint8)
            got = h.step(act, k=k)
            d_act[0].copy_(torch.from_numpy(act))
            d.step_device(d_act[0], d_obs[0], d_rew[0], d_done[0], k=k)
            want = device_out(1)
            same(got, (w[0] for w in want), (tag, "step k=%d" % k))

        act = rng.randint(2, size=(E, I)).astype(np.uint8)
        _, obs, rew, done = h.step_multi(3, actions=act, controller="given")
        d_act[0].copy_(torch.from_numpy(act))
        d.step_multi_device(3, d_act[0], d_obs, d_rew, d_done, controller="given")
        same((obs, rew, done), device_out(3), (tag, "step_multi given"))

        act_h, obs, rew, done = h.step_multi(3, controller="greedy", spacing=2)
        d.step_multi_device(3, d_act, d_obs, d_rew, d_done, controller="greedy", spacing=2)
        same((obs, rew, done), device_out(3), (tag, "step_multi greedy spacing 2"))
        assert act_h.tobytes() == d_act.cpu().numpy().tobytes(), (tag, "greedy actions")

        act = rng.randint(2, size=(E, I)).astype(np.uint8)
        mask = rng.rand(E) < 0.5
        h._obs[:] = -7.25                      # what the rows of the envs that are not stepped must keep
        h._reward[:] = 99.5
        h._done[:] = 7
        obs, rew, done = h.step_masked(act, mask, k=10)
        d_act[0].copy_(torch.from_numpy(act))
        d_mask = torch.from_numpy(mask.astype(np.uint8)).to(dev)
        check(d._L.te_step_masked(d._h, d_act[0].data_ptr(), d_mask.data_ptr(), 10, d_obs.data_ptr(), d_rew.data_ptr(),
                                  d_done.data_ptr(), TE_DEVICE, None))
        want = device_out(1)
        same((obs[mask], rew[mask], done[mask]), (w[0][mask] for w in want), (tag, "step_masked"))
        assert (obs[~mask] == np.float32(-7.25)).all() and (rew[~mask] == np.float32(99.5)).all() \
            and (done[~mask] == 7).all(), (tag, "step_masked: rows of envs not stepped")

        act = rng.randint(2, size=(E, I)).astype(np.uint8)
        h.step_wire(act, k=10)
        d_act[0].copy_(torch.from_numpy(act))
        check(d._L.te_step_wire(d._h, d_act[0].data_ptr(), 10, d_rec.data_ptr(), TE_DEVICE, None))
        d.synchronize()
        assert h._wire_buf[:, :done_at + 1].tobytes() == d_rec[0, :, :done_at + 1].cpu().numpy().tobytes(), (tag, "step_wire")

        act_h, _ = h.step_multi_wire(3, controller="greedy")    # one decision per launch again
        d._controller_spacing(None, 3, "greedy")
        check(d._L.te_step_multi_wire(d._h, 3, TE_CTRL_GREEDY, d_act[0].data_ptr(), 10, d_rec.data_ptr(), TE_DEVICE, None))
        d.synchronize()
        assert h._multi_wire[:3, :, :done_at + 1].tobytes() == d_rec[:, :, :done_at + 1].cpu().numpy().tobytes(), \
            (tag, "step_multi_wire")
        assert act_h.tobytes() == d_act[0].cpu().numpy().tobytes(), (tag, "step_multi_wire actions")
    assert h.stats()["vehicle_updates"] == d.stats()["vehicle_updates"] > 0
