"""Static objects that are Area polygons (containment counts) and a different map per scenario (t2d_set_map_polygons /
t2d_set_map_table), against the float64 oracle: flags, first-hit object and status bit-exact."""

import numpy as np
import pytest

from oracle import scenario as O
from tests.util import parking_like_objects

pytestmark = pytest.mark.gpu


def test_polygon_obstacles_containment_and_first_object(cuda_device):
    import torch

    from tactics2d_b200 import BatchedWorld, synthetic

    seg, ps = parking_like_objects()
    bounds = (-40.0, 40.0, -40.0, 40.0)
    n, m = 96, 16
    scene = synthetic.config2(n, m, seed=41, size=70.0)
    x = scene.x - 35.0
    y = scene.y - 35.0
    # hand-placed cases in scenario 0: deep inside the block (no edge in reach), inside the L's notch (inside its bounding
    # box, outside the polygon), on top of the small kerb stone (polygon inside the pose), straddling the wall, far away
    x[0, :5] = (-15.0, 8.0, 20.4, 0.0, 33.0)
    y[0, :5] = (-12.0, -10.0, 5.2, 18.5, 33.0)
    table = scene.table.as_oracle_table()
    w = BatchedWorld(n, m, scene.table, device=cuda_device, any_participant=True)
    w.set_map(seg, bounds, poly_start=ps)
    w.set_state(x, y, scene.heading, scene.speed, type_id=scene.type_id)
    r = w.check_events()
    torch.cuda.synchronize()
    fl, hi, hs = O.events(x, y, scene.heading, scene.type_id, table, seg, bounds, poly_start=ps)
    assert np.array_equal(r.flags.cpu().numpy(), fl)
    assert np.array_equal(r.hit_segment.cpu().numpy(), hs)
    assert np.array_equal(r.hit_index.cpu().numpy(), hi)
    # the hand-placed cases say what they were built to say
    assert hs[0, 0] == 4 and (fl[0, 0] & 2)          # wholly inside the block: object = its first segment
    assert hs[0, 1] == -1 and not (fl[0, 1] & 2)     # the notch of the L is free space
    assert hs[0, 2] == 14 and (fl[0, 2] & 2)         # the kerb stone under the car
    assert hs[0, 3] == 0 and (fl[0, 3] & 2)          # the wall
    assert hs[0, 4] == -1
    inside_only = 0
    plain = O.events(x, y, scene.heading, scene.type_id, table, seg, bounds)[0]
    inside_only = int((((fl & 2) != 0) & ((plain & 2) == 0)).sum())
    assert inside_only >= 10    # poses that only the containment rule catches
    # a few ticks: physics + events + status on the moving poses
    for t in range(3):
        act = torch.from_numpy(synthetic.random_actions(4100 + t, (n, m))).to(cuda_device)
        r = w.step(act)
        torch.cuda.synchronize()
        got = w.state_numpy()
        fl, hi, hs = O.events(got["x"], got["y"], got["heading"], scene.type_id, table, seg, bounds, poly_start=ps)
        assert np.array_equal(r.flags.cpu().numpy(), fl) and np.array_equal(r.hit_segment.cpu().numpy(), hs)
        st, done = O.status(fl, scene.type_id, np.full(n, t + 1), 0, ego_only=False)
        assert np.array_equal(r.status.cpu().numpy(), st)
    w.close()


def test_rejected_map_leaves_the_previous_map_in_force(cuda_device):
    """A set_map or set_map_table whose tile the compiler rejects changes nothing: the world keeps colliding with the map,
    and reading the tile ids, it had."""
    import torch

    from tactics2d_b200 import BatchedWorld, synthetic
    from tactics2d_b200._lib import T2DError

    seg, ps = parking_like_objects()
    bounds = (-40.0, 40.0, -40.0, 40.0)
    n, m = 32, 16
    scene = synthetic.config2(n, m, seed=47, size=70.0)
    x, y = scene.x - 35.0, scene.y - 35.0
    table = scene.table.as_oracle_table()
    w = BatchedWorld(n, m, scene.table, device=cuda_device, any_participant=True)
    w.set_map(seg, bounds, poly_start=ps)
    w.set_state(x, y, scene.heading, scene.speed, type_id=scene.type_id)
    fl, hi, hs = O.events(x, y, scene.heading, scene.type_id, table, seg, bounds, poly_start=ps)
    assert ((fl & 2) != 0).sum() > 0

    def check():
        r = w.check_events()
        torch.cuda.synchronize()
        assert np.array_equal(r.flags.cpu().numpy(), fl)
        assert np.array_equal(r.hit_segment.cpu().numpy(), hs) and np.array_equal(r.hit_index.cpu().numpy(), hi)

    check()
    open_ring = np.array([[0, 0, 4, 0], [4, 0, 4, 4], [4, 4, 0, 4], [0, 4, 0, 1]], np.float32)   # does not close
    with pytest.raises(T2DError, match="chain and close"):
        w.set_map(open_ring, (-10.0, 10.0, -10.0, 10.0), poly_start=[0, 4])
    check()
    # the same for a table: a rejected set_map_table keeps the previous tiles and the tile ids they are read with
    tiles = [dict(segments=seg, bounds=bounds, poly_start=ps), dict(segments=seg, bounds=(-30.0, 30.0, -30.0, 30.0), poly_start=None)]
    per_tile = [O.events(x, y, scene.heading, scene.type_id, table, t["segments"], t["bounds"], poly_start=t["poly_start"]) for t in tiles]
    ids = np.arange(n) % 2

    def expected(ids):
        return [np.where(ids[:, None] == 1, a1, a0) for a0, a1 in zip(*per_tile)]

    w.set_map_table(tiles, ids)
    fl, hi, hs = expected(ids)
    assert not np.array_equal(fl, expected(1 - ids)[0])
    check()
    with pytest.raises(T2DError, match="chain and close"):
        w.set_map_table([tiles[0], dict(segments=open_ring, bounds=None, poly_start=[0, 4])], 1 - ids)
    assert np.array_equal(w.tile_id.cpu().numpy(), ids)
    # id arrays of the same size allocated now would reuse the memory of a dropped one: they hold valid ids, the wrong ones
    filler = [torch.from_numpy((1 - ids).astype(np.int16)).to(cuda_device) for _ in range(4)]
    check()
    del filler
    w.close()


def test_map_table_one_tile_per_scenario(cuda_device):
    """configs[2] says "highD_map tiles": highD_1 .. highD_6 in ONE batch, every scenario on its own tile (segments and
    boundary box), plus a tile of polygons and an empty tile; tile ids rewritten between ticks."""
    import torch

    from tactics2d_b200 import BatchedWorld, synthetic
    from tactics2d_b200.map import load_collidable_segments

    tiles = []
    for k in range(1, 7):
        seg, bounds = load_collidable_segments(f"highD_{k}")
        tiles.append(dict(segments=seg, bounds=bounds, poly_start=None))
    pseg, ps = parking_like_objects()
    tiles.append(dict(segments=pseg, bounds=(-40.0, 40.0, -40.0, 40.0), poly_start=ps))
    tiles.append(dict(segments=None, bounds=(0.0, 100.0, -50.0, 50.0), poly_start=None))       # bounds only
    n, m = 64, 32
    rng = np.random.default_rng(5)
    tile_id = rng.integers(0, len(tiles), n)
    tile_id[:8] = np.arange(8)
    scene = synthetic.config3(n, m, seed=43, segments=None, bounds=tiles[0]["bounds"])
    x, y = scene.x.copy(), scene.y.copy()
    for s in range(n):
        b = tiles[tile_id[s]]["bounds"]
        x[s] = rng.uniform(b[0] - 3, b[1] + 3, m)
        y[s] = rng.uniform(b[2] - 3, b[3] + 3, m)
    table = scene.table.as_oracle_table()
    w = BatchedWorld(n, m, scene.table, device=cuda_device, any_participant=True)
    w.set_map_table(tiles, tile_id)
    w.set_state(x, y, scene.heading, scene.speed, type_id=scene.type_id)

    def check(r, xs, ys, hs_, ids):
        gfl, ghs, ghi = r.flags.cpu().numpy(), r.hit_segment.cpu().numpy(), r.hit_index.cpu().numpy()
        n_static = 0
        for s in range(n):
            t = tiles[ids[s]]
            fl, hi, hs = O.events(xs[s:s + 1], ys[s:s + 1], hs_[s:s + 1], scene.type_id[s:s + 1], table, t["segments"], t["bounds"],
                                  poly_start=t["poly_start"])
            assert np.array_equal(gfl[s], fl[0]), (s, ids[s])
            assert np.array_equal(ghs[s], hs[0]) and np.array_equal(ghi[s], hi[0]), (s, ids[s])
            n_static += int(((fl & 2) != 0).sum())
        return n_static

    r = w.check_events()
    torch.cuda.synchronize()
    assert check(r, x, y, scene.heading, tile_id) > 20
    for t in range(2):
        act = torch.from_numpy(synthetic.random_actions(4300 + t, (n, m), accel=(-6, 3), steer=(-0.05, 0.05))).to(cuda_device)
        r = w.step(act)
        torch.cuda.synchronize()
        got = w.state_numpy()
        check(r, got["x"], got["y"], got["heading"], tile_id)
    # a reset that draws new maps rewrites the ids in place: the next tick uses them
    new_ids = (tile_id + 3) % len(tiles)
    w.tile_id.copy_(torch.from_numpy(new_ids.astype(np.int16)))
    r = w.check_events()
    torch.cuda.synchronize()
    got = w.state_numpy()
    check(r, got["x"], got["y"], got["heading"], new_ids)
    # the lidar of a scenario sees its own tile's segments
    scan = w.lidar_scan(72, 30.0).cpu().numpy()
    for s in (0, 6, 7):
        t = tiles[new_ids[s]]
        w1 = BatchedWorld(1, m, scene.table, device=cuda_device)
        w1.set_map(t["segments"], t["bounds"], poly_start=t["poly_start"])
        w1.set_state(got["x"][s:s + 1], got["y"][s:s + 1], got["heading"][s:s + 1], got["speed"][s:s + 1], type_id=scene.type_id[s:s + 1])
        assert np.array_equal(w1.lidar_scan(72, 30.0).cpu().numpy()[0], scan[s])
        w1.close()
    w.close()


def test_log_seeded_reset_from_a_levelx_pool(cuda_device, tmp_path):
    """Log-seeded resets (SURVEY 8f rank 3): the pool ``initial_state_pool`` cuts out of a LevelX-schema log goes straight into
    ``t2d_reset``; the scenarios then tick from the logged states (empty slots stay empty)."""
    import torch

    from tactics2d_b200 import BatchedWorld
    from tactics2d_b200.dataset_parser import LevelXParser, initial_state_pool
    from tests.test_levelx_parser import _write_ind

    _write_ind(tmp_path)
    parser = LevelXParser("inD")
    pool, tid, table = initial_state_pool(parser, 3, str(tmp_path), 4, [0, 200, 360])
    n, m = 6, 4
    w = BatchedWorld(n, m, table, device=cuda_device, max_step=10)
    idx = np.array([0, 1, 2, 2, 1, 0], np.int32)
    w.type_id.copy_(torch.from_numpy(tid[idx]))
    dev_pool = {k: torch.from_numpy(v).to(cuda_device) for k, v in pool.items()}
    w.reset(torch.ones(n, dtype=torch.uint8, device=cuda_device), dev_pool, torch.from_numpy(idx).to(cuda_device))
    torch.cuda.synchronize()
    got = w.state_numpy()
    for k in ("x", "y", "heading", "speed", "vx", "vy"):
        assert np.array_equal(got[k], pool[k][idx]), k
    before = w.state_numpy()
    table_o = table.as_oracle_table()
    act = np.zeros((n, m, 2), np.float32)
    ref = O.physics_tick(before, tid[idx], act, table_o, 100, 5)
    w.step(torch.from_numpy(act).to(cuda_device))
    torch.cuda.synchronize()
    got = w.state_numpy()
    active = tid[idx] != 255
    assert active.sum() == 2 * (2 + 4 + 3)
    for k in ("x", "y", "speed"):
        assert np.max(np.abs(got[k] - ref[k])[active] / np.maximum(np.abs(ref[k][active]), 1.0)) <= 1e-5
    assert np.array_equal(got["x"][~active], before["x"][~active])
    w.close()


def test_worlds_of_different_size_interleave(cuda_device):
    """ADVICE r01: cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is per kernel and process-wide; a small world configured
    after a big one must not lower the big one's opt-in (tracked per device and kernel variant, only ever raised)."""
    import torch

    from tactics2d_b200 import BatchedWorld, synthetic
    from tactics2d_b200.map import load_collidable_segments

    seg, bounds = load_collidable_segments("rounD_0")       # a large tile: tens of KB of shared memory per CTA
    big = synthetic.config5(4096, 128, seed=51, segments=seg, bounds=bounds)       # 8 warps per CTA, big map
    small = synthetic.config2(8, 16, seed=52, size=40.0)                           # 2 warps per CTA, tiny map
    wb = BatchedWorld(*big.shape, big.table, device=cuda_device)
    wb.set_map(big.segments, big.bounds)
    wb.set_state(big.x, big.y, big.heading, big.speed, type_id=big.type_id)
    ws = BatchedWorld(*small.shape, small.table, device=cuda_device)
    ws.set_map(small.segments, small.bounds)
    ws.set_state(small.x, small.y, small.heading, small.speed, type_id=small.type_id)
    ab = torch.zeros((*big.shape, 2), device=cuda_device)
    as_ = torch.zeros((*small.shape, 2), device=cuda_device)
    table_b, table_s = big.table.as_oracle_table(), small.table.as_oracle_table()
    for _ in range(2):
        for w, a, sc, tb in ((wb, ab, big, table_b), (ws, as_, small, table_s), (wb, ab, big, table_b)):
            r = w.step(a)
            torch.cuda.synchronize()
            got = w.state_numpy()
            sel = slice(0, 8)
            fl, hi, hs = O.events(got["x"][sel], got["y"][sel], got["heading"][sel], sc.type_id[sel], tb, sc.segments, sc.bounds)
            assert np.array_equal(r.flags.cpu().numpy()[sel], fl) and np.array_equal(r.hit_segment.cpu().numpy()[sel], hs)
    wb.close(); ws.close()


def test_masked_reset_starts_wheel_speeds_and_last_accel_fresh(cuda_device):
    """ADVICE r01: a masked reset re-initialises ALL per-participant state the world owns: the SingleTrackDrift wheel speeds
    (pool columns, or free rolling speed / wheel_radius) and the controllers' State.accel of the previous tick (0)."""
    import torch

    from tactics2d_b200 import BatchedWorld, TypeParams, TypeTable
    from tactics2d_b200.controller import AccelerationController

    n, m = 6, 8
    table = TypeTable([TypeParams.vehicle("medium_car", model="drift")])
    w = BatchedWorld(n, m, table, device=cuda_device)
    z = np.zeros((n, m), np.float32)
    speed = np.full((n, m), 6.0, np.float32)
    w.set_state(z, z, z, speed, type_id=np.zeros((n, m), np.uint8))
    w.set_wheel_state(speed / 0.344, speed / 0.344)
    cid = np.zeros((n, m), np.uint8)
    w.set_controllers([AccelerationController(12.0)], cid)
    act = torch.zeros((n, m, 2), device=cuda_device)
    for _ in range(3):
        w.control(act); w.step(act)
    torch.cuda.synchronize()
    assert float(w.last_accel.abs().max()) > 0 and not torch.allclose(w.omega_front, torch.from_numpy(speed / 0.344).to(cuda_device))
    mask = torch.tensor([1, 0, 1, 0, 0, 1], dtype=torch.uint8, device=cuda_device)
    pool = {k: torch.from_numpy(v).to(cuda_device) for k, v in dict(x=z, y=z, heading=z, speed=np.full((n, m), 4.0, np.float32)).items()}
    before = (w.omega_front.clone(), w.omega_rear.clone(), w.last_accel.clone())
    w.reset(mask, pool)
    torch.cuda.synchronize()
    mb = mask.bool()
    wr = float(np.float32(4.0) / np.float32(table.rows[0].wheel_radius))
    assert torch.allclose(w.omega_front[mb], torch.full_like(w.omega_front[mb], wr)) and torch.allclose(w.omega_rear[mb], torch.full_like(w.omega_rear[mb], wr))
    assert float(w.last_accel[mb].abs().max()) == 0.0
    assert torch.equal(w.omega_front[~mb], before[0][~mb]) and torch.equal(w.last_accel[~mb], before[2][~mb])     # untouched scenarios
    pool["omega_wf"] = torch.full((n, m), 9.0, device=cuda_device)
    pool["omega_wr"] = torch.full((n, m), 8.0, device=cuda_device)
    w.reset(mask, pool)
    torch.cuda.synchronize()
    assert float(w.omega_front[mb].min()) == 9.0 and float(w.omega_rear[mb].max()) == 8.0
    # arguments that would be raw-pointer accidents are rejected on the host
    with pytest.raises(ValueError):
        w.reset(torch.ones(n + 1, dtype=torch.uint8, device=cuda_device), pool)
    with pytest.raises(ValueError):
        w.reset(mask, {**pool, "x": pool["x"].cpu()})
    w.reset(mask.cpu(), pool)          # a host mask is moved, not dereferenced on the device
    torch.cuda.synchronize()
    w.close()
