"""risk_check_initial_backup_trajectory (the initial-backup-trajectory check of the start pool) through the ABI export list,
the config and the command line; no GPU."""
from safemotionsrisk_b200 import abi
from safemotionsrisk_b200.cli import env_config_from_command
from safemotionsrisk_b200.config import EnvConfig

RISK = dict(risk_config_dir="risk_networks/state_action/space", risk_threshold=0.065)


def test_new_symbols_are_in_the_export_list():
    for sym in ("smenv_set_initial_backup_check", "smenv_initial_backup_check_counts"):
        assert sym in abi.EXPORTED_SYMBOLS


def test_config_accepts_the_flag_with_the_networks():
    cfg = EnvConfig(risk_check_initial_backup_trajectory=True, **RISK)
    assert cfg.risk_check_initial_backup_trajectory is True
    cfg = EnvConfig(risk_check_initial_backup_trajectory=True, risk_state_initial_backup_trajectory_steps=12, **RISK)
    assert cfg.risk_state_initial_backup_trajectory_steps == 12


def test_cli_flag_pastes_through():
    cfg = env_config_from_command(
        "python safemotions/train.py --risk_config_dir=risk_networks/state_action/space --risk_threshold=0.065 "
        "--risk_check_initial_backup_trajectory --risk_state_initial_backup_trajectory_steps=20")
    assert cfg.risk_check_initial_backup_trajectory is True
    assert cfg.risk_state_initial_backup_trajectory_steps == 20
    assert cfg.risk_config_dir == "risk_networks/state_action/space" and cfg.risk_threshold == 0.065
