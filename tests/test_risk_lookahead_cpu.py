"""risk_state_config 4 (the backup-trajectory look-ahead inside the step) through the config and the command line; no GPU."""
import pytest

from safemotionsrisk_b200.cli import env_config_from_command
from safemotionsrisk_b200.config import EnvConfig

RISK = dict(risk_config_dir="risk_networks/state_action/space", risk_threshold=0.065)


def test_config_4_is_accepted_with_the_networks_and_a_threshold():
    cfg = EnvConfig(risk_state_config=4, **RISK)
    assert cfg.risk_state_config == 4
    assert EnvConfig(risk_state_config=4, risk_state_backup_trajectory_steps=12, **RISK).risk_state_backup_trajectory_steps == 12


def test_config_4_needs_risk_config_dir():
    with pytest.raises(ValueError):
        EnvConfig(risk_state_config=4)
    with pytest.raises(ValueError):
        EnvConfig(risk_state_config=4, risk_threshold=0.065)
    with pytest.raises(ValueError):   # risk_config_dir without a threshold, as for the network gate
        EnvConfig(risk_state_config=4, risk_config_dir=RISK["risk_config_dir"])


@pytest.mark.parametrize("value", [1, 2, 3])
def test_forecasting_configs_still_raise(value):
    with pytest.raises(NotImplementedError):
        EnvConfig(risk_state_config=value, **RISK)


def test_cli_flag_selects_config_4():
    cfg = env_config_from_command(
        "python safemotions/train.py --risk_config_dir=risk_networks/state_action/space --risk_threshold=0.065 "
        "--risk_state_config=RISK_CHECK_NEXT_STATE_SIMULATE_NEXT_STEP_AND_BACKUP_TRAJECTORY "
        "--risk_state_backup_trajectory_steps=20")
    assert cfg.risk_state_config == 4
    assert cfg.risk_state_backup_trajectory_steps == 20
    assert cfg.risk_config_dir == "risk_networks/state_action/space" and cfg.risk_threshold == 0.065
