"""CLI: `check -i` report and the launcher command builder / single-node launch (reference: colossalai/cli)."""
import os
import subprocess
import sys
import tempfile

from colossalai_b200.cli import cli
from colossalai_b200.cli.launcher.run import fetch_hostfile, get_launch_command, parse_device_filter

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_check_report(capsys):
    assert cli(["check", "-i"]) == 0
    out = capsys.readouterr().out
    assert "Installation Report" in out and "sm_100a" in out


def test_launch_command_and_hostfile():
    cmd = get_launch_command("127.0.0.1", 29511, 4, "train.py", ["--lr", "1"], extra_launch_args="max_restarts=0")
    assert "torch.distributed.run" in cmd and "--nproc_per_node=4" in cmd and cmd.endswith("train.py --lr 1")
    multi = get_launch_command("node0", 29511, 8, "train.py", [], node_rank=1, num_nodes=2)
    assert "--rdzv_endpoint=node0:29511" in multi and "--node_rank=1" in multi
    with tempfile.NamedTemporaryFile("w", suffix=".txt", delete=False) as f:
        f.write("hostA\nhostB\n# comment\nhostC\n")
    pool = fetch_hostfile(f.name, None)
    assert len(pool) == 3
    assert [h.hostname for h in parse_device_filter(pool, exclude_str="hostB")] == ["hostA", "hostC"]
    os.unlink(f.name)


def test_run_single_node(tmp_path):
    script = tmp_path / "hello.py"
    script.write_text("import os\nopen(os.environ['OUT'] + os.environ['RANK'], 'w').write(os.environ['WORLD_SIZE'])\n")
    env = dict(os.environ, OUT=str(tmp_path / "rank"), PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, "-m", "colossalai_b200", "run", "--nproc_per_node", "2", "--master_port",
                        "29617", str(script)], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert (tmp_path / "rank0").read_text() == "2" and (tmp_path / "rank1").read_text() == "2"
