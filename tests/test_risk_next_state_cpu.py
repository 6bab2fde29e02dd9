"""risk_state_config 3 (rate the simulated next state with a state risk network) through the config and the command line;
no GPU."""
import pytest

from safemotionsrisk_b200.cli import env_config_from_command
from safemotionsrisk_b200.config import EnvConfig

STATE_DIR = "results/state_risk/space/20260101T000000"   # where risk_train writes a state network


def test_config_3_is_accepted_with_a_state_network_dir_and_a_threshold():
    cfg = EnvConfig(risk_state_config=3, risk_config_dir=STATE_DIR, risk_threshold=0.3)
    assert cfg.risk_state_config == 3 and cfg.risk_config_dir == STATE_DIR


def test_config_3_is_accepted_with_an_npz_path():
    cfg = EnvConfig(risk_state_config=3, risk_config_dir="/tmp/nets/state_net.npz", risk_threshold=0.3)
    assert cfg.risk_state_config == 3


def test_config_3_needs_the_network_and_a_threshold():
    with pytest.raises(ValueError):
        EnvConfig(risk_state_config=3)
    with pytest.raises(ValueError):
        EnvConfig(risk_state_config=3, risk_threshold=0.3)
    with pytest.raises(ValueError):
        EnvConfig(risk_state_config=3, risk_config_dir=STATE_DIR)


@pytest.mark.parametrize("path", ["risk_networks/state_action/space", "results/state_action_risk/space/20260101T000000",
                                  "results/state_action_risk/space/20260101T000000/risk_network.npz"])
def test_config_3_with_a_state_action_network_is_not_implemented(path):
    with pytest.raises(NotImplementedError):
        EnvConfig(risk_state_config=3, risk_config_dir=path, risk_threshold=0.065)


@pytest.mark.parametrize("value", [1, 2])
def test_forecasting_configs_raise(value):
    with pytest.raises(NotImplementedError):
        EnvConfig(risk_state_config=value, risk_config_dir=STATE_DIR, risk_threshold=0.3)


def test_cli_flag_selects_config_3():
    cfg = env_config_from_command(
        "python safemotions/train.py --risk_config_dir={} --risk_threshold=0.3 "
        "--risk_state_config=RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP".format(STATE_DIR))
    assert cfg.risk_state_config == 3
    assert cfg.risk_config_dir == STATE_DIR and cfg.risk_threshold == 0.3
