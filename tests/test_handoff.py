"""Device-resident engine -> parser hand-off behind the reference's host-only feature_map_t (csrc/handoff.h; SURVEY 8f-2).

The operator API sequence (examples/operator_api_batched_images_paf.example.cpp:64-74) is
    packets = engine.inference(batch); for packet in packets: parser.process(packet[0], packet[1])
with every tensor crossing host memory.  The drop-in keeps the interface; these tests pin the behaviour behind it:
  * buffers the engine filled AND published are parsed once per batch from the device snapshot (counters prove it),
    results byte-identical to the oracle and to the ordinary host path;
  * anything else -- a copy at another address, ANY changed byte, a publication older than 4 batches, the switch
    turned off -- takes the host path and gives the same answer."""
import os
import threading

import numpy as np
import pytest

import oracle
from hyperpose_b200 import capi, models, synthetic as syn
from tests.golden.make_golden import pifpaf_handoff_case, sha

pytestmark = pytest.mark.gpu


def _engine_with_synthetic_outputs(N, seed=3, persons=(2, 4)):
    """tiny network whose conf/paf outputs are overwritten (bench hook) with synthetic skeleton tensors: every conv still
    runs, and the parser has people to find"""
    import torch
    H, W = 64, 96
    eng = capi.Engine(models.tiny_test_net(4).to_pack(), (W, H), max_batch_size=N)
    conf, paf = syn.make_batch_tensors(seed, N, persons, eng.out_h, eng.out_w)
    dc, dp = torch.from_numpy(conf).cuda(), torch.from_numpy(paf).cuda()
    torch.cuda.synchronize()
    eng.set_output_override(dc.data_ptr(), dp.data_ptr())
    frames = syn.make_frames_u8(9, N, H, W)
    return eng, frames, conf, paf, (dc, dp)


def _delta(before):
    now = capi.handoff_stats()
    return {k: now[k] - before[k] for k in now}


def test_published_batch_is_parsed_once_on_the_device():
    N = 4
    eng, frames, conf, paf, keep = _engine_with_synthetic_outputs(N)
    parser = capi.PafParser()
    eng.infer_u8(frames)
    s0 = capi.handoff_stats()
    packets = eng.read_outputs_frames(N, publish=True)                      # tensorrt::inference's return value
    assert _delta(s0)["published"] == 1
    l0 = parser.launch_count
    total = 0
    for i, (c, p) in enumerate(packets):
        assert c.tobytes() == conf[i].tobytes() and p.tobytes() == paf[i].tobytes()
        got = parser.process(c, p)                            # paf::process(packet[0], packet[1])
        want = oracle.oracle_process(conf[i], paf[i])["humans"]
        assert got.tobytes() == want.tobytes(), f"frame {i}"
        total += len(got)
    d = _delta(s0)
    assert d["hits"] == N and d["batch_parses"] == 1 and d["misses"] == 0, d
    assert parser.launch_count - l0 == 2, "one batched launch sequence (2 kernels) for the whole batch"
    assert total >= N, "vacuous: no humans in the synthetic tensors"
    # the same buffers again (a second parser.process on a packet): still served from the cached batch
    again = parser.process(packets[1][0], packets[1][1])
    assert again.tobytes() == oracle.oracle_process(conf[1], paf[1])["humans"].tobytes()
    assert _delta(s0)["batch_parses"] == 1
    eng.close(); parser.close()


def test_copies_changed_contents_and_other_parameters():
    N = 3
    eng, frames, conf, paf, keep = _engine_with_synthetic_outputs(N, seed=5)
    parser = capi.PafParser()
    eng.infer_u8(frames)
    packets = eng.read_outputs_frames(N, publish=True)
    # (a) a copy at another address is not a published buffer: ordinary host path, same answer
    s0 = capi.handoff_stats()
    c2, p2 = packets[0][0].copy(), packets[0][1].copy()
    assert parser.process(c2, p2).tobytes() == oracle.oracle_process(conf[0], paf[0])["humans"].tobytes()
    assert _delta(s0)["hits"] == 0
    # (b) other thresholds on the published buffers: the batch is parsed again with them
    s0 = capi.handoff_stats()
    parser.set_conf_thresh(0.3); parser.set_paf_thresh(0.1)
    for i in range(N):
        want = oracle.oracle_process(conf[i], paf[i], 0.3, 0.1)["humans"]
        assert parser.process(*packets[i]).tobytes() == want.tobytes()
    d = _delta(s0)
    assert d["hits"] == N and d["batch_parses"] == 1, d
    # (c) contents changed behind the API's back -- ONE float somewhere in the middle of either tensor (the look-up compares every
    #     byte with the published copy, not a sample): host path on the new bytes, never the cached humans of the old ones
    for which, idx, delta in ((0, (7, 13, 21), 0.5), (1, (29, 5, 40), -0.75)):
        s0 = capi.handoff_stats()
        saved = float(packets[2][which][idx])
        packets[2][which][idx] += delta
        want = oracle.oracle_process(packets[2][0], packets[2][1], 0.3, 0.1)["humans"]
        assert parser.process(*packets[2]).tobytes() == want.tobytes()
        d = _delta(s0)
        assert d["hits"] == 0 and d["misses"] == 1, d
        packets[2][which][idx] = saved                          # restored bytes are the published bytes again: served from the cache
        s0 = capi.handoff_stats()
        assert parser.process(*packets[2]).tobytes() == oracle.oracle_process(conf[2], paf[2], 0.3, 0.1)["humans"].tobytes()
        assert _delta(s0)["hits"] == 1
    # (d) switched off: nothing is published, nothing is looked up
    capi.handoff_enable(False)
    try:
        s0 = capi.handoff_stats()
        eng.infer_u8(frames)
        pk = eng.read_outputs_frames(N, publish=True)
        parser.set_conf_thresh(0.05); parser.set_paf_thresh(0.05)
        for i in range(N):
            assert parser.process(*pk[i]).tobytes() == oracle.oracle_process(conf[i], paf[i])["humans"].tobytes()
        d = _delta(s0)
        assert d["published"] == 0 and d["hits"] == 0, d
    finally:
        capi.handoff_enable(True)
    eng.close(); parser.close()


def test_old_publications_are_retired_and_engine_teardown_unregisters():
    N = 2
    eng, frames, conf, paf, keep = _engine_with_synthetic_outputs(N, seed=7)
    parser = capi.PafParser()
    batches = []
    for _ in range(5):                                        # ring of 4: the first publication is retired by the fifth
        eng.infer_u8(frames)
        batches.append(eng.read_outputs_frames(N, publish=True))
    s0 = capi.handoff_stats()
    want = [oracle.oracle_process(conf[i], paf[i])["humans"].tobytes() for i in range(N)]
    for i in range(N):
        assert parser.process(*batches[0][i]).tobytes() == want[i]
    assert _delta(s0)["hits"] == 0
    for i in range(N):
        assert parser.process(*batches[4][i]).tobytes() == want[i]
    assert _delta(s0)["hits"] == N
    eng.close()                                               # snapshots freed, addresses unregistered
    s0 = capi.handoff_stats()
    for i in range(N):
        assert parser.process(*batches[3][i]).tobytes() == want[i]
    assert _delta(s0)["hits"] == 0
    parser.close()


def test_stream_style_parser_replicas_on_threads():
    """the stream's parse stage (stream.hpp:347-373): one thread-pool task per image, each on its own parser replica"""
    N = 6
    eng, frames, conf, paf, keep = _engine_with_synthetic_outputs(N, seed=11)
    eng.infer_u8(frames)
    packets = eng.read_outputs_frames(N, publish=True)
    replicas = [capi.PafParser() for _ in range(N)]
    got = [None] * N
    s0 = capi.handoff_stats()

    def task(i):
        got[i] = replicas[i].process(*packets[i])

    th = [threading.Thread(target=task, args=(i,)) for i in range(N)]
    [t.start() for t in th]
    [t.join() for t in th]
    for i in range(N):
        assert got[i].tobytes() == oracle.oracle_process(conf[i], paf[i])["humans"].tobytes()
    d = _delta(s0)
    assert d["hits"] == N and d["batch_parses"] == 1, d
    for r in replicas:
        r.close()
    eng.close()


def test_pifpaf_fields_hand_off(golden_dir):
    import torch
    N, HW = 2, 385
    eng = capi.Engine(models.resnet50_pifpaf(0).to_pack(), (HW, HW), max_batch_size=N)
    assert eng.head_type == 1 and (eng.out_h, eng.out_w) == (49, 49)
    live = np.load(os.path.join(golden_dir, "ref_live.npz"))      # what the reference decoder (oracle/_ref) returned on these fields
    pif, paf = pifpaf_handoff_case()
    assert sha(pif) + sha(paf) == str(live["pp_handoff_in_sha"]), "synthetic generator drifted from the goldens"
    dp, da = torch.from_numpy(pif).cuda(), torch.from_numpy(paf).cuda()
    torch.cuda.synchronize()
    eng.set_output_override(dp.data_ptr(), da.data_ptr())
    eng.infer_u8(syn.make_frames_u8(1, N, HW, HW))
    s0 = capi.handoff_stats()
    packets = eng.read_outputs_frames(N, publish=True)                      # [pif_i [17,5,49,49], paf_i [19,9,49,49]]
    dec = capi.PifPafParser(HW, HW, 0.1)
    total = 0
    for i in range(N):
        assert packets[i][0].shape == (17, 5, 49, 49) and packets[i][0].tobytes() == pif[i].tobytes()
        got = dec.process(packets[i][0], packets[i][1])
        want = live[f"pp_handoff{i}_humans"]
        if oracle.pifpaf_ref_available():
            assert oracle.ref_pifpaf_process(pif[i], paf[i], HW, HW, 0.1).tobytes() == want.tobytes()
        assert got.tobytes() == want.tobytes(), (i, len(got), len(want))
        total += len(got)
    d = _delta(s0)
    assert d["hits"] == N and d["batch_parses"] == 1, d
    assert total >= N
    dec.close(); eng.close()
