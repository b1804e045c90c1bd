"""GPU test of the C++ adapter classes (cn_chess_ai_b200/adapter/xq_adapter.hpp): the reference's ChessBoard /
ChessAI / DQN / Action API surface, driven the way MainWindow/Worker drive the originals."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_exe(tmp_path):
    exe = tmp_path / "test_adapter"
    pkg = os.path.join(ROOT, "cn_chess_ai_b200")
    subprocess.run(["g++", "-std=c++17", "-O1", "-o", str(exe), os.path.join(ROOT, "tests", "cpp", "test_adapter.cpp"), "-L" + pkg,
                    "-lxq_b200", "-Wl,-rpath," + pkg], check=True)
    return exe


def test_cpp_adapter_transcript(tmp_path, O):
    exe = build_exe(tmp_path)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    got = dict((ln.split()[0], ln.split()[1:]) for ln in out.stdout.strip().splitlines())
    # known answers of the reference (SURVEY section 4, re-derived from the unmodified build when it is present)
    want = {"opening_actions": ["44", "first", "0", "9"], "valid_2_1_9_1": ["1", "valid_0_0_5_5", "0"],
            "captured": ["4", "1", "red_score", "40", "eval", "39", "-40", "37"],
            "moves_9_0": ["3", "player", "1", "movecount", "1", "over", "0"], "copy_movecount": ["0", "orig_movecount", "1"],
            "state": ["1260", "ones", "31"], "q_size": ["8100", "q_in_range", "1"], "trained_games": ["1", "red_score_nonneg", "1", "dqn", "1"],
            "ai_move_valid": ["1"], "ai_move_other_colour_valid": ["12"], "ai_move_sentinel": ["-1", "-1", "-1", "-1"],
            "nn_sizes": ["50", "9", "offsets", "0", "30", "0", "5"],
            "nn_init_ok": ["1", "1", "trained", "1", "host_untouched", "1", "host_changed", "1", "copy_from_equal", "1", "copy_ctor_equal", "1"],
            "batched_games": ["300", "last", "300", "finished", "1", "report", "300", "updates_positive", "1"]}
    for k, v in want.items():
        assert got[k] == v, (k, got[k], v)
    assert out.stdout.count("invalid_argument") == 3 and out.stdout.count("runtime_error") == 1
    log = (tmp_path / "game_log.txt").read_text().splitlines()
    assert len(log) == 302 and log[0].startswith("Game 1 completed. Red Score: ") and log[300] == "AI self-play session completed. Total games: 300"
    R = O.ref()
    if R is not None:   # the same calls through the reference's own classes
        h = C.c_void_p(R.ref_env_new())
        buf = np.zeros(256, np.int32)
        assert R.ref_env_all_actions(h, 0, buf) == 44 and R.ref_env_is_valid_move(h, 2, 1, 9, 1) == 1
        assert R.ref_env_move(h, 19, 82) == 11 and R.ref_env_evaluate(h, 0, 1) == 39 and R.ref_env_evaluate(h, 1, 1) == -40
        assert R.ref_env_valid_moves(h, 9, 0, buf) == 3


@pytest.mark.parametrize("mode", ["trainparity", "selfplayparity"])
def test_cpp_chessai_train_equals_the_reference_chessai_train(tmp_path, O, make_golden, answers, mode):
    """The drop-in claim end to end: `ChessAI::train(2)` / `ChessAI::startSelfPlay(2)` (src/chessai.cpp:191-266) of the C++ adapter (every device operation through the C ABI: legal lists, selectAction,
    movePiece, state, FP64 forward / TD step as written, target sync) against the reference's OWN `ChessAI::train(2)` (unmodified
    sources) started from the same model file and fed the same rand() stream: same gameCompleted events, final weights equal to 1e-10.
    The reference's result is stored in tests/golden/reference_answers.npz; with oracle/_ref built it is also run live."""
    import cn_chess_ai_b200 as xq
    w, b, stream = make_golden.adapter_inputs()
    net = xq.DQN([1260, 128, 8100])
    net.set_params(w, b)
    net.save_model(tmp_path / "in.bin")
    exe = build_exe(tmp_path)
    out = subprocess.run([str(exe), mode, str(tmp_path / "in.bin"), "2", str(tmp_path / "out.bin")], capture_output=True, text=True,
                         timeout=900, cwd=str(tmp_path))
    assert out.returncode == 0, out.stderr[-2000:]
    ev_gpu = [int(v) for ln in out.stdout.splitlines() if ln.startswith("event ") for v in ln.split()[1:]]
    net.load_model(tmp_path / "out.bin")
    w_gpu, b_gpu = net.get_params()
    net.close()
    key = "adapter_train" if mode == "trainparity" else "adapter_selfplay"
    assert ev_gpu == list(answers[key + "_events"]) and len(ev_gpu) == 6
    assert int(answers[key + "_consumed"]) <= len(stream)
    make_golden.check_loop(answers, key, w, b, stream, w_gpu, b_gpu, 1e-10)
    assert np.abs(w_gpu - w).max() > 1e-6
    R = O.ref()
    if R is None:
        return
    h = C.c_void_p(R.ref_env_new())
    R.ref_rand_load(stream, len(stream))
    w_ref, b_ref = np.zeros_like(w), np.zeros_like(b)
    P = C.c_void_p
    ref_run = R.ref_ai_train if mode == "trainparity" else R.ref_ai_selfplay
    cwd = os.getcwd()
    os.chdir(tmp_path)                       # the reference's startSelfPlay / onGameCompleted append to game_log.txt in the working directory
    try:
        assert ref_run(h, 2, w.ctypes.data_as(P), b.ctypes.data_as(P), w_ref.ctypes.data_as(P), b_ref.ctypes.data_as(P)) == 0
    finally:
        os.chdir(cwd)
    assert R.ref_rand_consumed() <= len(stream)
    ev_ref = np.zeros(3 * R.ref_events_count(), np.int32)
    R.ref_events_get(ev_ref)
    R.ref_env_free(h)
    assert ev_gpu == list(ev_ref) and len(ev_gpu) == 6
    assert np.abs(w_gpu - w_ref).max() < 1e-10 and np.abs(b_gpu - b_ref).max() < 1e-10
