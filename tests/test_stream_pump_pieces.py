"""The multi-stream side of the streaming pump (dbeel_b200/csrc/host/stream_pump.h: publish_pieces, end_at), the flow
of the streamed hash-range scan, on a box without a GPU and under ThreadSanitizer when the toolchain has it
(tests/stream_pump_pieces_test.cc)."""
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "stream_pump_pieces_test.cc")


def _tsan_works(tmp_path):
    probe = tmp_path / "probe.cc"
    probe.write_text("#include <thread>\nint main() { std::thread t([] {}); t.join(); return 0; }\n")
    exe = str(tmp_path / "probe")
    if subprocess.run(["g++", "-fsanitize=thread", "-pthread", str(probe), "-o", exe], capture_output=True).returncode:
        return False
    return subprocess.run([exe], capture_output=True).returncode == 0


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_stream_pump_pieces_every_byte_once_end_and_errors(tmp_path):
    exe = str(tmp_path / "stream_pump_pieces_test")
    flags = ["-O1", "-g", "-fsanitize=thread"] if _tsan_works(tmp_path) else ["-O2"]
    subprocess.check_call(["g++", *flags, "-std=c++17", "-pthread", SRC, "-o", exe])
    env = dict(os.environ, TSAN_OPTIONS="halt_on_error=1 exitcode=66")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=500, env=env)
    assert out.returncode == 0, out.stdout + out.stderr[-4000:]
    assert out.stdout.strip().endswith("ok")
