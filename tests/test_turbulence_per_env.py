"""CPU: the boundary of the per-env Fried parameter -- validation, the r0 -> sqrt(Cn^2) conversion, and how a reset
option reaches the library (a recording stand-in for the device handle)."""
import numpy as np
import pytest


def test_validation_rejects_bad_values():
    from adaptive_optics_gym_b200.env import fried_values
    from adaptive_optics_gym_b200.tables import FRIED_MIN
    good = [0.05, 0.10, 0.20, 0.08]
    vals, scalar = fried_values(good, 4)
    assert vals.dtype == np.float64 and vals.tolist() == good and not scalar
    for bad, match in (([0.1, 0.1, 0.1], 'one per env'), ([[0.1, 0.1], [0.1, 0.1]], 'one per env'),
                       ([0.1, np.nan, 0.1, 0.1], 'finite'), ([0.1, np.inf, 0.1, 0.1], 'finite'),
                       ([0.1, 0.0, 0.1, 0.1], 'positive'), ([0.1, -0.2, 0.1, 0.1], 'positive'),
                       ([0.1, 0.1, 0.999 * FRIED_MIN, 0.1], '>='), (np.nan, 'finite'), (0.005, '>=')):
        with pytest.raises(ValueError, match=match):
            fried_values(bad, 4)
    assert fried_values(FRIED_MIN, 4)[0].tolist() == [FRIED_MIN] * 4


def test_constructor_validates_before_any_device_call():
    pytest.importorskip('torch')
    from adaptive_optics_gym_b200 import AOVecEnv
    for bad in ([0.1, 0.2], [0.1, 0.2, float('nan'), 0.1], [0.1, 0.2, 0.003, 0.1]):
        with pytest.raises(ValueError):
            AOVecEnv(4, atm_fried=bad)


def test_per_element_conversion_equals_scalar_conversion():
    """env i of a per-env handle must use, bit for bit, the sqrt(Cn^2) of a handle built with the scalar r0_i
    (env.py: ``c.sqrt_cn2 = float(np.sqrt(cn2_from_fried(float(atm_fried), wavelength_sci)))``)."""
    from adaptive_optics_gym_b200.tables import AOConfig, cn2_from_fried, sqrt_cn2_from_fried
    wl = AOConfig().wavelength_sci
    r0 = np.exp(np.random.default_rng(0).uniform(np.log(0.01), np.log(0.5), 4096))
    got = sqrt_cn2_from_fried(r0, wl)
    want = np.array([float(np.sqrt(cn2_from_fried(float(r), wl))) for r in r0.tolist()])
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    # the same from a tuple
    assert np.array_equal(sqrt_cn2_from_fried(tuple(r0.tolist()), wl), got)


class _RecordingHandle:
    def __init__(self):
        self.calls = []

    def set_turbulence(self, sqrt_cn2, rescale=False, stream=None):
        self.calls.append((np.array(sqrt_cn2), rescale))


def _bare_env(atm_type, num_envs=4):
    from adaptive_optics_gym_b200.env import _AOCore
    from adaptive_optics_gym_b200.tables import AOConfig
    env = _AOCore()
    env.num_envs, env.atm_type = num_envs, atm_type
    env.wavelength_sci = AOConfig().wavelength_sci
    env.fried_parameter = 0.15
    env._h = _RecordingHandle()
    return env


def test_reset_option_broadcasts_a_scalar_and_picks_the_rescale():
    from adaptive_optics_gym_b200.tables import sqrt_cn2_from_fried
    env = _bare_env('quasi_static')
    env._reset_options({'atm_fried': 0.1})
    (v, rescale), = env._h.calls
    assert rescale and v.tolist() == sqrt_cn2_from_fried([0.1] * 4, env.wavelength_sci).tolist()
    assert isinstance(env.fried_parameter, float) and env.fried_parameter == 0.1
    env._reset_options({'atm_fried': np.array([0.05, 0.1, 0.2, 0.08])})
    assert env._h.calls[-1][1] and isinstance(env.fried_parameter, np.ndarray)
    assert env.fried_parameter.tolist() == [0.05, 0.1, 0.2, 0.08]
    # semi_dynamic stores the values: the reset's new screens are drawn at them
    env = _bare_env('semi_dynamic')
    env._reset_options({'atm_fried': [0.05, 0.1, 0.2, 0.08]})
    assert env._h.calls[-1][1] is False
    # no option, another option, or an invalid value: nothing reaches the library
    env = _bare_env('dynamic')
    for opts in (None, {}, {'other': 1}):
        env._reset_options(opts)
    with pytest.raises(ValueError):
        env._reset_options({'atm_fried': [0.1, 0.1]})
    assert env._h.calls == [] and env.fried_parameter == 0.15


def test_reset_option_takes_a_tensor():
    torch = pytest.importorskip('torch')
    env = _bare_env('dynamic')
    env._reset_options({'atm_fried': torch.tensor([0.05, 0.1, 0.2, 0.08], dtype=torch.float64)})
    assert env.fried_parameter.tolist() == [0.05, 0.1, 0.2, 0.08] and env._h.calls[-1][1]
