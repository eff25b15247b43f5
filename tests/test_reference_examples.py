"""The reference's OWN example programs -- /root/reference/examples/*.cpp compiled UNMODIFIED against the drop-in (the
north star: "drops into the existing C++ examples unchanged") -- build here and run on the GPU box.

Build (hyperpose_b200/build.py::build_reference_examples): every source is compiled where it lies in the reference tree --
the example, examples/utils.cpp, and the reference's own src/{stream,thread_pool,logging,human,data}.cpp (scheduler,
draw_human, non_scaling_resize) -- over the unchanged public headers, with the B200 classes of csrc/hyperpose_api underneath
and the OpenCV / gflags stand-ins of csrc/shim (neither library exists in this image).  The binaries land in
oracle/_ref/dropin/ref_build/, with the other builds of the reference's sources.

Inputs: the shim's only image container is binary PPM, so the "images" are P6 files named *.png and the "video" is P6 frames
back to back; model files are HPB2PACK packs named as the example expects (.onnx where it insists on that suffix)."""
import os
import subprocess

import numpy as np
import pytest

from hyperpose_b200 import build as hb, models, synthetic as syn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _p6(frame_bgr: np.ndarray) -> bytes:
    h, w, _ = frame_bgr.shape
    return b"P6\n%d %d\n255\n" % (w, h) + np.ascontiguousarray(frame_bgr[..., ::-1]).tobytes()


def _read_p6_stream(path):
    data = open(path, "rb").read()
    frames, pos = [], 0
    while pos < len(data):
        assert data[pos:pos + 2] == b"P6", data[pos:pos + 16]
        parts, p = [], pos + 2
        while len(parts) < 3:
            while data[p:p + 1].isspace():
                p += 1
            q = p
            while not data[q:q + 1].isspace():
                q += 1
            parts.append(int(data[p:q]))
            p = q
        w, h, _ = parts
        p += 1
        frames.append(np.frombuffer(data[p:p + w * h * 3], np.uint8).reshape(h, w, 3)[..., ::-1])
        pos = p + w * h * 3
    return frames


def _exes():
    exes = hb.build_reference_examples()
    if exes is None:
        pytest.skip("reference examples not built (they need the reference's sources at build time)")
    return exes


def test_reference_examples_build_unmodified_against_the_dropin():
    exes = _exes()
    assert len(exes) == 6
    for name, exe in exes.items():
        assert os.path.exists(exe), name
    syms = subprocess.run(["nm", "-C", "--defined-only", exes["cli"]], capture_output=True, text=True).stdout
    # the reference's own scheduler / drawing code is in the binary, over the B200 engine and parsers
    for want in ["hyperpose::basic_stream_manager::write_to(cv::VideoWriter&)", "hyperpose::draw_human(cv::Mat&",
                 "hyperpose::non_scaling_resize(", "hyperpose::dnn::tensorrt::inference(std::vector<cv::Mat", "hyperpose::parser::paf::process(",
                 "hyperpose::parser::pifpaf::process(", "hyperpose::parser::pose_proposal::process("]:
        assert want in syms, want
    und = subprocess.run(["nm", "-C", "--undefined-only", exes["cli"]], capture_output=True, text=True).stdout
    assert "hp_engine_create" in und and "hp_paf_process_host" in und      # reached through the C ABI of libhyperpose_b200.so
    # gflags stand-in: flags parse, unknown flags are fatal
    r = subprocess.run([exes["gen_serialized_engine.example"], "--no_such_flag=1"], capture_output=True, text=True)
    assert r.returncode == 1 and "unknown command line flag" in r.stderr


def _write_inputs(tmp_path, n, h, w, seed=5):
    folder = tmp_path / "media"
    folder.mkdir()
    frames = syn.make_frames_u8(seed, n, h, w)
    for i in range(n):
        (folder / f"img_{i:02d}.png").write_bytes(_p6(frames[i]))
    video = tmp_path / "video.avi"
    video.write_bytes(b"".join(_p6(f) for f in frames))
    return folder, video, frames


@pytest.mark.gpu
def test_operator_api_batched_images_paf_example_runs(tmp_path):
    """examples/operator_api_batched_images_paf.example.cpp:58-74, unmodified"""
    exes = _exes()
    folder, _, _ = _write_inputs(tmp_path, 3, 80, 112)            # frames larger than the network: engine-side resize runs
    pack = tmp_path / "tiny.pack"
    pack.write_bytes(models.tiny_test_net(0).to_pack())
    r = subprocess.run([exes["operator_api_batched_images_paf.example"], f"--model_file={pack}", f"--input_folder={folder}", "--input_width=96", "--input_height=64"],
                       capture_output=True, text=True, timeout=180, cwd=tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "3 images got processed" in r.stdout and r.stdout.count("conf:[19, 32, 48, ]") == 3
    outs = sorted(p for p in os.listdir(tmp_path) if p.startswith("output_"))
    assert outs == ["output_0.png", "output_1.png", "output_2.png"]
    img = _read_p6_stream(tmp_path / "output_0.png")[0]
    assert img.shape == (64, 96, 3)                               # cv::resize(batch[i], batch[i], {w, h}) before drawing (example :79)


@pytest.mark.gpu
def test_operator_api_batched_images_pifpaf_example_runs(tmp_path):
    """examples/operator_api_batched_images_pifpaf.example.cpp:48-64, unmodified"""
    exes = _exes()
    folder, _, _ = _write_inputs(tmp_path, 2, 129, 129)
    pack = tmp_path / "pifpaf.pack"
    pack.write_bytes(models.resnet50_pifpaf(0).to_pack())
    r = subprocess.run([exes["operator_api_batched_images_pifpaf.example"], f"--model_file={pack}", f"--input_folder={folder}", "--input_width=129", "--input_height=129"],
                       capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "2 images got processed" in r.stdout


@pytest.mark.gpu
def test_stream_api_video_paf_example_runs(tmp_path):
    """examples/stream_api_video_paf.example.cpp:80-95, unmodified: hp::make_stream(engine, parser); stream.async() << capture;
    stream.sync() >> writer -- the reference's own scheduler threads over the B200 engine / parser, video in, video out"""
    exes = _exes()
    _, video, frames = _write_inputs(tmp_path, 11, 64, 96)
    pack = tmp_path / "tiny.pack"
    pack.write_bytes(models.tiny_test_net(0).to_pack())
    out = tmp_path / "out.avi"
    r = subprocess.run([exes["stream_api_video_paf.example"], f"--model_file={pack}", f"--input_video={video}", f"--output_video={out}",
                        "--input_width=96", "--input_height=64", "--max_batch_size=4"], capture_output=True, text=True, timeout=180, cwd=tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "11 images got processed" in r.stdout
    written = _read_p6_stream(out)
    assert len(written) == 11 and written[0].shape == (64, 96, 3)


@pytest.mark.gpu
def test_gen_serialized_engine_example_runs(tmp_path):
    """examples/gen_serialized_engine.example.cpp:28-46, unmodified: tensorrt(onnx{...}).save(path); the saved file loads through
    tensorrt_serialized{path} (the paf example takes any non-.onnx/.uff name that way)"""
    exes = _exes()
    model = tmp_path / "tiny.onnx"                                # the example insists on an .onnx / .uff suffix
    model.write_bytes(models.tiny_test_net(0).to_pack())
    saved = tmp_path / "tiny.trt"
    r = subprocess.run([exes["gen_serialized_engine.example"], f"--model_file={model}", f"--output_model={saved}", "--input_width=96", "--input_height=64", "--max_batch_size=2"],
                       capture_output=True, text=True, timeout=120, cwd=tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    assert saved.read_bytes() == model.read_bytes()
    folder, _, _ = _write_inputs(tmp_path, 2, 64, 96)
    r = subprocess.run([exes["operator_api_batched_images_paf.example"], f"--model_file={saved}", f"--input_folder={folder}", "--input_width=96", "--input_height=64"],
                       capture_output=True, text=True, timeout=180, cwd=tmp_path)
    assert r.returncode == 0 and "2 images got processed" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("runtime,source", [("operator", "folder"), ("operator", "video"), ("stream", "video")])
def test_cli_runs(tmp_path, runtime, source):
    """examples/cli.cpp, unmodified: parser std::variant (:39-54), operator runtime on an image folder / a video, stream runtime"""
    exes = _exes()
    folder, video, frames = _write_inputs(tmp_path, 5, 64, 96)
    pack = tmp_path / "tiny.pack"
    pack.write_bytes(models.tiny_test_net(0).to_pack())
    src = folder if source == "folder" else video
    r = subprocess.run([exes["cli"], f"--model={pack}", "--w=96", "--h=64", "--max_batch_size=2", f"--source={src}", f"--runtime={runtime}", "--post=paf",
                        "--imshow=false", f"--saving_prefix={tmp_path / 'out'}"], capture_output=True, text=True, timeout=180, cwd=tmp_path)
    assert r.returncode == 0, r.stdout + r.stderr
    # the stream runtime prints basic_stream_manager::processed_num() = m_ingest, which the reference increments once more for the
    # empty frame that ends the video (src/stream.cpp:50-52): 6 for a 5-frame video, with real OpenCV as well
    assert ("6 images got processed" if runtime == "stream" else "5 images got processed") in r.stdout, r.stdout
    if source == "folder":
        assert len([p for p in os.listdir(tmp_path) if p.startswith("out_") and p.endswith(".png")]) == 5
    else:
        assert len(_read_p6_stream(tmp_path / "out.avi")) == 5
