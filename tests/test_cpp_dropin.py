"""The C++ drop-in (hyperpose::parser::paf / hyperpose::dnn::tensorrt over the C ABI):
  * CPU: compiles and links against the reference's UNCHANGED public headers (when /root/reference exists);
  * GPU: the prebuilt example binary runs the reference's operator-API sequence end to end."""
import os
import subprocess

import pytest

from hyperpose_b200 import build as hb, models

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(not os.path.isdir("/root/reference/include/hyperpose"), reason="reference headers absent")
def test_dropin_compiles_against_unchanged_reference_headers():
    exe = os.path.join(hb.REF_BIN, "operator_api_b200")
    if os.path.exists(exe):
        os.remove(exe)
    assert hb.build_cpp_example() == exe and os.path.exists(exe)
    syms = subprocess.run(["nm", "-C", "--defined-only", exe], capture_output=True, text=True).stdout
    for want in ["hyperpose::parser::paf::process(", "hyperpose::parser::paf::paf(float, float, cv::Size)",
                 "hyperpose::parser::paf::set_conf_thresh(float)", "hyperpose::dnn::tensorrt::inference(std::vector<cv::Mat",
                 "hyperpose::dnn::tensorrt::inference(std::vector<float", "hyperpose::dnn::tensorrt::save(", "hyperpose::parser::pifpaf::process(",
                 "hyperpose::parser::pose_proposal::process(", "hyperpose::parser::pose_proposal::set_nms_thresh(float)"]:
        assert want in syms, want


@pytest.mark.gpu
def test_cpp_example_runs_operator_api_sequence(tmp_path):
    exe = hb.build_cpp_example()
    if exe is None:
        pytest.skip("example binary not built (needs the reference headers at build time)")
    pack = tmp_path / "tiny.pack"
    pack.write_bytes(models.tiny_test_net(0).to_pack())
    saved = tmp_path / "saved.pack"
    r = subprocess.run([exe, str(pack), "96", "64", "3", str(saved)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert saved.read_bytes() == pack.read_bytes()      # tensorrt::save re-emits the pack
    assert "conf:[19, 32, 48, ]" in r.stdout and "paf:[38, 32, 48, ]" in r.stdout
    assert "3 images got processed" in r.stdout
    # several batches: the parser calls of a batch are served from the device snapshot the engine published
    # (csrc/handoff.h); with the hand-off disabled the same program prints the same human counts
    a = subprocess.run([exe, str(pack), "96", "64", "3", "-", "3"], capture_output=True, text=True, timeout=120)
    b = subprocess.run([exe, str(pack), "96", "64", "3", "-", "3"], capture_output=True, text=True, timeout=120,
                       env=dict(os.environ, HPB_NO_HANDOFF="1"))
    assert a.returncode == 0 and b.returncode == 0, a.stderr + b.stderr
    counts = lambda out: [ln.split("humans = ")[1] for ln in out.splitlines() if "humans = " in ln]
    assert len(counts(a.stdout)) == 3 and counts(a.stdout) == counts(b.stdout)


@pytest.mark.gpu
def test_cpp_example_pifpaf_sequence(tmp_path):
    """examples/operator_api_batched_images_pifpaf.example.cpp:48-64: packets come back ordered by name (paf < pif) with
    rank-4 shapes, which is what pifpaf::process(packet[0], packet[1]) expects (src/pifpaf.cpp:6-7)"""
    exe = hb.build_cpp_example()
    if exe is None:
        pytest.skip("example binary not built (needs the reference headers at build time)")
    pack = tmp_path / "pifpaf.pack"
    pack.write_bytes(models.resnet50_pifpaf(0).to_pack())
    r = subprocess.run([exe, str(pack), "129", "129", "2", "-", "2", "pifpaf"], capture_output=True, text=True, timeout=180)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "paf:[19, 9, 17, 17, ] pif:[17, 5, 17, 17, ]" in r.stdout
    assert r.stdout.count("2 images got processed") == 2


def test_reference_stream_scheduler_builds_over_the_dropin_and_runs_with_a_mock_engine():
    """SURVEY 8f-2: `hyperpose::make_stream(engine, parser)` (include/hyperpose/stream/stream.hpp:311-319) with the reference's
    own scheduler sources (src/stream.cpp, src/thread_pool.cpp) compiled unchanged:
      * instantiates and links over the B200 `tensorrt` / `paf` classes (examples/stream_api_b200);
      * the same program with a stand-in engine / parser (no GPU) runs the scheduler end to end: every frame reaches the sink,
        the poses drawn equal the operator-API count, the stream shuts down."""
    exe, mock = hb.build_stream_example(), hb.build_stream_example(mock=True)
    if exe is None or mock is None:
        pytest.skip("stream example binaries not built (need the reference sources at build time)")
    syms = subprocess.run(["nm", "-C", "--defined-only", exe], capture_output=True, text=True).stdout
    assert "hyperpose::basic_stream_manager::resize_from_inputs(cv::Size)" in syms
    assert "hyperpose::stream<hyperpose::dnn::tensorrt, hyperpose::parser::paf>" in syms
    for n, mb in ((37, 4), (200, 8), (1, 1)):
        r = subprocess.run([mock, "-", "96", "64", str(mb), str(n)], capture_output=True, text=True, timeout=60)
        assert r.returncode == 0, r.stdout + r.stderr
        assert f"{n} frames through the stream" in r.stdout and "stream == operator API" in r.stdout


@pytest.mark.gpu
def test_reference_stream_scheduler_runs_on_the_gpu(tmp_path):
    exe = hb.build_stream_example()
    if exe is None:
        pytest.skip("example binary not built (needs the reference sources at build time)")
    pack = tmp_path / "tiny.pack"
    pack.write_bytes(models.tiny_test_net(0).to_pack())
    r = subprocess.run([exe, str(pack), "96", "64", "4", "12"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "12 frames through the stream" in r.stdout and "stream == operator API" in r.stdout
