"""make_env is a drop-in for rlschool.make_env('Quadrupedal', ...) (ETGRL/train.py:305-309): every keyword it cannot honour must
raise NotImplementedError BEFORE any device work (VERDICT r1 weak #8 / ADVICE r1: no silent kwarg swallowing)."""
import numpy as np
import pytest


def _mk(**kw):
    from paddlerobotics_b200.env import make_env
    return make_env("Quadrupedal", **kw)


@pytest.mark.parametrize("kw", [dict(render=True), dict(task="cave"), dict(task="gallop"), dict(sensor_mode={"footpose": 1}), dict(sensor_mode={"dynamic_vec": 1}),
                                dict(sensor_mode={"force_vec": 1}), dict(sensor_mode={"ETG_obs": 1}), dict(sensor_mode={"lidar": 1}),
                                dict(sensor_mode={"RNN": {"mode": "GRU", "time_steps": 5, "time_interval": 1}}),
                                dict(motor_control_mode=4), dict(motor_control_mode="PWM"), dict(random_param={"random_terrain": 1}), dict(ETG_H=30),
                                dict(reward_param={"stand": 0.5})])
def test_unsupported_keywords_raise(kw):
    with pytest.raises(NotImplementedError):
        _mk(**kw)


def test_other_env_names_raise():
    from paddlerobotics_b200.env import make_env
    with pytest.raises(NotImplementedError):
        make_env("Quadrotor")


def test_unknown_keyword_is_a_type_error_not_ignored():
    with pytest.raises((TypeError, RuntimeError)):
        _mk(task="ground", no_such_option=1)


def test_terrain_presets_follow_the_reference_parameters():
    """train.py:48-50: STEP_HEIGHT 0.08..0.10, SLOPE 0.2..0.4, STEP_WIDTH 0.26..0.40; every reference task name that is provided
    builds, starts flat around the reset pose and reaches n_steps*step_height at the top."""
    from paddlerobotics_b200 import terrain as T
    assert np.isclose(T.STEP_HEIGHT[0], 0.08) and np.isclose(T.STEP_HEIGHT[-1], 0.10) and np.isclose(T.SLOPE[0], 0.2) and np.isclose(T.SLOPE[-1], 0.4)
    assert np.isclose(T.STEP_WIDTH[0], 0.26) and np.isclose(T.STEP_WIDTH[-1], 0.40)
    assert T.make_terrain("ground") is None and T.make_terrain("plane") is None
    for task in ("stairstair", "stairslope", "slopestair", "slopeslope"):
        for sh in (0.08, 0.10):
            hf, x0, y0, cell = T.make_terrain(task, step_height=sh, step_width=0.26, slope=0.4, n_steps=4)
            xs = x0 + cell * np.arange(hf.shape[1])
            assert np.all(hf[:, (xs > -0.5) & (xs < 0.7)] == 0.0)                   # flat where the robot is reset (x_noise +-0.1)
            assert np.isclose(hf.max(), 4 * sh) and hf[0, -1] == 0.0 and np.all(hf == hf[0:1])
            if task.startswith("stair"):
                up = hf[0][(xs > 0.8) & (xs < 0.8 + 4 * 0.26)]
                assert set(np.round(np.unique(up) / sh).astype(int)) <= {1, 2, 3, 4}    # treads at whole multiples of step_height
    bb, x0, y0, cell = T.make_terrain("balancebeam", step_y=0.05)
    ys = y0 + cell * np.arange(bb.shape[0])
    assert bb[np.abs(ys) < 0.1][:, -1].max() == 0.0 and bb[np.abs(ys) > 0.3][:, -1].max() == -0.3
    with pytest.raises(NotImplementedError):
        T.make_terrain("cave")
    p = T.sample_terrain_params(np.random.default_rng(0))
    assert 0.08 <= p["step_height"] <= 0.1001 and 0.2 <= p["slope"] <= 0.4001 and 0.26 <= p["step_width"] <= 0.4001
