"""ldpcsim --error-log argument handling; nothing here needs a GPU (the log file is opened before the code is loaded)."""
import os
import subprocess

from conftest import H_FILE, ROOT

CLI = os.path.join(ROOT, "libldpc_b200", "ldpcsim")


def test_error_log_arguments(built_lib, tmp_path):
    r = subprocess.run([CLI, "--help"], capture_output=True, text=True)
    assert r.returncode == 0 and "--error-log" in r.stdout
    r = subprocess.run([CLI, H_FILE, str(tmp_path / "o.txt"), "-5", "-4", "0.5", "--error-log"], capture_output=True, text=True)
    assert r.returncode != 0 and "Too few arguments for '--error-log'" in r.stdout
    bad = tmp_path / "no_such_dir" / "err.log"
    r = subprocess.run([CLI, H_FILE, str(tmp_path / "o.txt"), "-5", "-4", "0.5", "--error-log", str(bad)], capture_output=True, text=True)
    assert r.returncode != 0 and "--error-log: cannot open" in r.stdout
    assert not (tmp_path / "o.txt").exists()
