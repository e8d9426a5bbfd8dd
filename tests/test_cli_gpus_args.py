"""The --gpus flag of ``python -m idelucs_b200`` (no GPU needed): the combinations the data-parallel path does not take are
rejected with a one-line parser error naming the flag, and without --gpus (or with --gpus 1) the argument dictionary handed
to run() is exactly the reference CLI's."""
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


@pytest.mark.parametrize("extra", [[], ["--gpus", "1"]], ids=["no_flag", "gpus_1"])
def test_single_gpu_args_unchanged(calls, extra):
    cli.main(["--sequence_file", "x.fas"] + extra)
    assert calls == [("run", REFERENCE_ARGS)]


def test_multi_gpu_dispatch(calls):
    cli.main(["--sequence_file", "x.fas", "--gpus", "4", "--n_clusters", "5", "--optimizer", "Adam"])
    assert calls == [("run_gpus", dict(REFERENCE_ARGS, n_clusters=5, optimizer="Adam"), 4)]


@pytest.mark.parametrize("argv,flag", [
    (["--gpus", "2", "--batch_sz", "255"], "--batch_sz"),
    (["--gpus", "4", "--batch_sz", "258"], "--batch_sz"),
    (["--gpus", "2", "--model_size", "small"], "--model_size"),
    (["--gpus", "2", "--model_size", "full"], "--model_size"),
    (["--gpus", "2", "--scheduler", "Plateau"], "--scheduler"),
    (["--gpus", "2", "--scheduler", "Triangle"], "--scheduler"),
    (["--gpus", "2", "--optimizer", "Adagrad"], "--optimizer"),
    (["--gpus", "8"], "--gpus"),
    (["--gpus", "0"], "--gpus"),
    (["--gpus", "-2"], "--gpus"),
], ids=["batch_odd", "batch_not_multiple_of_4", "small", "full", "plateau", "triangle", "optimizer", "too_many_gpus", "zero", "negative"])
def test_rejected_with_parser_error(calls, capsys, argv, flag):
    with pytest.raises(SystemExit) as e:
        cli.main(["--sequence_file", "x.fas"] + argv)
    assert e.value.code == 2
    err = [line for line in capsys.readouterr().err.splitlines() if line.startswith("idelucs: error:")]
    assert len(err) == 1 and flag in err[0], err
    assert calls == []
