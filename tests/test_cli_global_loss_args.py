"""The --global_batch_loss flag of ``python -m idelucs_b200`` (no GPU needed): with --gpus N >= 2 it reaches the data-parallel
path as args["global_batch_loss"]; with one GPU (which already trains on the global batch) it is accepted and dropped; without it
the argument dictionary is exactly the reference CLI's."""
import pytest

torch = pytest.importorskip("torch")

from idelucs_b200 import __main__ as cli   # noqa: E402

REFERENCE_ARGS = {"sequence_file": "x.fas", "n_clusters": 0, "n_epochs": 100, "n_mimics": 3, "batch_sz": 256, "GT_file": None, "k": 6,
                  "optimizer": "RMSprop", "scheduler": "None", "weight": 0.25, "lambda": 2.8, "lr": 1e-3, "n_voters": 5,
                  "model_size": "linear", "plot": False}


@pytest.fixture
def calls(monkeypatch):
    got = []
    monkeypatch.setattr(cli, "run", lambda args: got.append(("run", dict(args))))
    monkeypatch.setattr(cli, "run_gpus", lambda args, gpus: got.append(("run_gpus", dict(args), gpus)))
    monkeypatch.setattr(torch.cuda, "device_count", lambda: 4)
    return got


def test_multi_gpu_dispatch_with_global_loss(calls):
    cli.main(["--sequence_file", "x.fas", "--gpus", "4", "--global_batch_loss", "--n_clusters", "5"])
    assert calls == [("run_gpus", dict(REFERENCE_ARGS, n_clusters=5, global_batch_loss=True), 4)]


@pytest.mark.parametrize("extra", [["--gpus", "1", "--global_batch_loss"], ["--global_batch_loss"]], ids=["gpus_1", "no_gpus_flag"])
def test_single_gpu_drops_the_flag(calls, extra):
    cli.main(["--sequence_file", "x.fas"] + extra)
    assert calls == [("run", REFERENCE_ARGS)]


@pytest.mark.parametrize("extra", [[], ["--gpus", "1"], ["--gpus", "2"]], ids=["no_flag", "gpus_1", "gpus_2"])
def test_without_the_flag_nothing_changes(calls, extra):
    cli.main(["--sequence_file", "x.fas"] + extra)
    assert calls == ([("run_gpus", REFERENCE_ARGS, 2)] if extra[-1:] == ["2"] else [("run", REFERENCE_ARGS)])


def test_flag_takes_no_value(calls, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(["--sequence_file", "x.fas", "--gpus", "2", "--global_batch_loss=1"])
    assert e.value.code == 2 and calls == []
    assert "--global_batch_loss" in capsys.readouterr().err
