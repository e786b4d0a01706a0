"""bench.py --impl reference: the reference arm runs the UNMODIFIED reference on torch CPU and prints one JSON line with the
contract's keys.  Without the reference files (oracle/_ref, made by build() where the reference is installed) the arm times
the numpy oracle port instead and says so in the line."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    sys.path.insert(0, ROOT)
    from oracle.ref_loader import reference_root
    have_reference = reference_root() is not None
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "mel_frames_per_sec_100step_ddpm" and line["value"] > 0
    assert line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["higher_is_better"] is True
    if have_reference:
        assert line["cpu_baseline"]["kind"] == "reference"
        assert "unmodified reference" in line["cpu_baseline"]["sample"]
    else:
        assert line["cpu_baseline"]["kind"] == "port"
        assert "numpy oracle port" in line["cpu_baseline"]["sample"]
