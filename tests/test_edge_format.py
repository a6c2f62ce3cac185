"""The reduced-set edge format rule (csrc/edge_fmt.cuh), checked on the host: working sets of at most 65 536 points
get 4-byte edges (i << 16 | j), larger ones 8-byte edges, and the arena takes that many bytes per edge."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
CUDA_INC = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


def test_edge_format_follows_the_working_set_size(tmp_path):
    exe = str(tmp_path / "edge_fmt_snippet")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I", CUDA_INC, "-I", CSRC, "-x", "c++",
                           os.path.join(ROOT, "tests", "cpp", "edge_fmt_snippet.cc"), "-o", exe])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=60)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "edge format ok" in r.stdout
