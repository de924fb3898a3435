"""Host side of playing against a frozen network, without a GPU: the command lines of the trainer and of the evaluation,
and loading an opponent from every format Agent(base_net_file=...) accepts."""
import pytest
import torch


def test_training_cli_opponent_options():
    from azul_deep_reinforcement_learning_b200.train import parse_args
    a = parse_args(["256", "run1", "--opponent", "old.pt", "--opponent-refresh", "10"])
    assert (a.batch_size, a.net_name, a.opponent, a.opponent_refresh) == (256, "run1", "old.pt", 10)
    b = parse_args([])
    assert b.opponent is None and b.opponent_refresh == 0
    with pytest.raises(SystemExit):
        parse_args(["--opponent-refresh", "-1"])


def test_evaluate_cli():
    from azul_deep_reinforcement_learning_b200.evaluate import MODES, parse_args
    a = parse_args(["net.pt"])
    assert (a.net, a.opponent, a.games, a.mode, a.seed) == ("net.pt", "random", 2048, "sample", 0)
    b = parse_args(["net.pt", "--opponent", "old.mx", "--games", "4096", "--mode", "argmax", "--seed", "7"])
    assert (b.opponent, b.games, MODES[b.mode], b.seed) == ("old.mx", 4096, 1, 7)
    for bad in (["net.pt", "--mode", "greedy"], ["net.pt", "--games", "0"], []):
        with pytest.raises(SystemExit):
            parse_args(bad)


def test_opponent_loads_from_every_saved_format(tmp_path):
    """A state dict, the trainer's checkpoint (object or file), a pickled ActorCritic and a module all give the same
    parameters; anything else is refused."""
    from azul_deep_reinforcement_learning_b200.azulnet.model import ActorCritic
    from azul_deep_reinforcement_learning_b200.selfplay import load_network
    torch.manual_seed(12)
    net = ActorCritic(136, 180)
    want = {k: v.clone() for k, v in net.state_dict().items()}
    ckpt = {"ac_net": net.state_dict(), "optimizer": torch.optim.Adam(net.parameters()).state_dict(), "batch": 3}
    torch.save(net.state_dict(), str(tmp_path / "bare.pt"))
    torch.save(ckpt, str(tmp_path / "ckpt.pt"))
    torch.save(net, str(tmp_path / "module.mx"))
    for src in (net.state_dict(), ckpt, net, str(tmp_path / "bare.pt"), str(tmp_path / "ckpt"), tmp_path / "module.mx"):
        got = load_network(src).state_dict()
        assert set(got) == set(want) and all(torch.equal(got[k], want[k]) for k in want), type(src)
    with pytest.raises(TypeError):
        load_network(42)
    with pytest.raises(FileNotFoundError):
        load_network(str(tmp_path / "missing"))
