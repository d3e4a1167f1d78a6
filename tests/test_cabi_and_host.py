"""CPU-side checks (no GPU): the C-ABI library loads and exports every symbol include/rlctr.h
declares, ctypes struct layouts match the header, and the host logic (fused-row layout, reference-keyed
state_dict, Adam schedule, init RNG order) behaves like the reference."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from oracle import torch_port as TP

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from rl_ctr_prediction_b200 import _lib, build
    if not os.path.exists(_lib.LIB_PATH):
        build.build()
    return _lib.load()


def header_symbols():
    text = open(os.path.join(ROOT, "include", "rlctr.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(rlctr_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    from rl_ctr_prediction_b200 import _lib
    syms = header_symbols()
    assert len(syms) >= 18
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/rlctr.h but not exported"
    assert set(syms) == set(_lib.SIGNATURES), set(syms) ^ set(_lib.SIGNATURES)
    assert lib.rlctr_version() == 100
    assert lib.rlctr_strerror(-1) == b"invalid argument"


def test_struct_layouts_match_header(tmp_path):
    """ctypes mirrors of the C structs: sizes and key offsets equal what gcc computes from include/rlctr.h itself."""
    import subprocess
    from rl_ctr_prediction_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rlctr.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(rlctr_table), sizeof(rlctr_adam), sizeof(rlctr_rowgrad), offsetof(rlctr_table,row_stride),'
                   'offsetof(rlctr_adam,sched_len), offsetof(rlctr_table,peers), offsetof(rlctr_rowgrad,peer_staged),'
                   'offsetof(rlctr_rowgrad,peer_extra), offsetof(rlctr_adam,stage), sizeof(rlctr_lookup),'
                   'offsetof(rlctr_lookup,gathered));return 0;}\n')
    exe = tmp_path / "layout"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_lib.Table), C.sizeof(_lib.Adam), C.sizeof(_lib.RowGrad), _lib.Table.row_stride.offset,
            _lib.Adam.sched_len.offset, _lib.Table.peers.offset, _lib.RowGrad.peer_staged.offset, _lib.RowGrad.peer_extra.offset,
            _lib.Adam.stage.offset, C.sizeof(_lib.Lookup), _lib.Lookup.gathered.offset]
    assert got == want, (got, want)
    assert C.sizeof(_lib.Table) == 104 and C.sizeof(_lib.Adam) == 88 and C.sizeof(_lib.RowGrad) == 304


def test_member_struct_layout_matches_header(tmp_path):
    """struct rlctr_member (co-located records) as gcc lays it out == the ctypes mirror."""
    import subprocess
    from rl_ctr_prediction_b200 import _lib
    src = tmp_path / "member.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rlctr.h"\nint main(void){printf("%zu %zu %zu %zu %zu %d\\n",'
                   'sizeof(rlctr_member), offsetof(rlctr_member,bias), offsetof(rlctr_member,pctr_stride),'
                   'offsetof(rlctr_member,rows_pitch), offsetof(rlctr_member,extra), RLCTR_GROUP_MAX);return 0;}\n')
    exe = tmp_path / "member"
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.run(["gcc", "-I", os.path.join(root, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    want = [C.sizeof(_lib.Member), _lib.Member.bias.offset, _lib.Member.pctr_stride.offset, _lib.Member.rows_pitch.offset,
            _lib.Member.extra.offset, _lib.RLCTR_GROUP_MAX]
    assert got == want, (got, want)


def test_colocated_layout_rules():
    """colocated._layout: vector members keep their stand-alone chunk alignment, scalar members take padding columns, the stamp
    gets a free column of the last active chunk, and the joint row stays within one 128-byte line."""
    from rl_ctr_prediction_b200 import colocated, tables, _lib

    class M:
        def __init__(self, g):
            self._geom = g
    lr, fm = (lambda: M(tables.Geometry.lr(100))), (lambda d=10: M(tables.Geometry.fm(100, d)))
    cols, used = colocated._layout([lr(), fm(), fm()])                      # LR + FM + DeepFM, D = 10
    assert cols == [(11, 0, 0), (0, 1, 10), (12, 13, 10)] and used == 23    # LR's weight in FM's padding column, stamp at 23
    cols, used = colocated._layout([fm(), lr(), lr(), fm()])
    assert cols == [(0, 1, 10), (11, 0, 0), (23, 0, 0), (12, 13, 10)] and used == 25      # no free column left: a dummy, then the stamp
    cols, used = colocated._layout([fm(11), lr()])                          # a full 12-float block: LR opens a new chunk
    assert cols == [(0, 1, 11), (12, 0, 0)] and used == 13
    for c, _ in [colocated._layout([fm(), fm()]), colocated._layout([lr()])]:
        assert all(e % 4 == 1 for _, e, d in c if d)                        # latent columns start at 1 mod 4, as stand-alone
    with pytest.raises(_lib.RlctrError):
        colocated._layout([fm(), fm(), fm()])                               # 36 + stamp floats: wider than one line
    with pytest.raises(_lib.RlctrError):
        colocated._layout([M(tables.Geometry.ffm(100, 15, 10))])


def test_argument_errors_need_no_gpu(lib):
    # argument validation happens before any CUDA call
    assert lib.rlctr_embed_fwd(None, None, None, None, None, 1, None, None, 0, 4, 15, 1, None) == -1
    assert lib.rlctr_generate_preds(None, None, None, None, None, None, None, 4, 3, 0, None) == -1
    assert lib.rlctr_generate_preds_v10(None, None, None, None, None, None, None, None, 4, 3, None, 0, None) == -1
    assert lib.rlctr_generate_preds_v10_ws_bytes(1000) >= 4 * 8 * 4
    assert lib.rlctr_rows_catchup_ids(None, 4, None, None, None, 0, None) == -1
    assert lib.rlctr_rows_claim_bytes(1000) == 32 * 4 and lib.rlctr_rows_claim_bytes(0) == 0
    assert lib.rlctr_sort_ids(None, 1, 1, None, None, None, 0, None) == -1
    assert lib.rlctr_rows_ws_bytes(1000) >= 16
    assert lib.rlctr_group_fwd(None, None, None, 0, None, 0, 4, 15, None) != 0
    assert lib.rlctr_group_rows_adam(None, None, 4, None, None, None, 1, None, 0, 15, 1, None, None, 0, None) == -1
    assert lib.rlctr_push_rows_routed(None, 4, 2, 0, 8, None, 10, None, None) == -1
    assert lib.rlctr_sort_routed_pos(None, 4, 10, None, None, None, 0, None) == -1


@pytest.mark.parametrize("name", ["LR", "FM", "FFM", "DeepFM"])
def test_state_dict_is_reference_keyed_and_init_matches_seed(name):
    """Same torch.manual_seed => same initial parameters as the reference-ordered constructors, and
    state_dict()/load_state_dict() speak the reference's keys and shapes (SURVEY section 8b)."""
    from rl_ctr_prediction_b200 import pretrain_main as PM
    N, F, D = 50, 15, 10
    torch.manual_seed(1)
    port = TP.PortCTR(name, N, F, D)
    torch.manual_seed(1)
    m = PM.get_model(name, N, F, D)
    sd, ref = m.state_dict(), port.state_dict()
    assert set(sd.keys()) == set(ref.keys())
    for k in ref:
        assert tuple(sd[k].shape) == tuple(ref[k].shape), k
        assert torch.equal(sd[k], ref[k]), k
    # load a perturbed checkpoint back
    ref2 = {k: v + 1 for k, v in ref.items()}
    m.load_state_dict(ref2)
    for k, v in m.state_dict().items():
        assert torch.equal(v, ref2[k])
    with pytest.raises(RuntimeError):
        m.load_state_dict({k: v for k, v in ref2.items() if k != "linear.weight"})
    # pad columns stay zero
    g = m._geom
    used = torch.zeros(g.row_stride, dtype=torch.bool)
    if g.lin_col >= 0:
        used[g.lin_col] = True
    used[g.emb_col:g.emb_col + g.dim] = True
    assert torch.all(m.table.data[:, :g.row_stride][:, ~used] == 0)
    # trainable tables carry Adam's exp_avg / exp_avg_sq inside each row record, zero until an optimizer runs
    assert g.row_pitch == (4 if g.row_stride == 1 else 3 * g.row_stride) and m.table.shape[1] == g.row_pitch   # LR: [w|m|v|stamp]
    assert torch.all(m.table.data[:, g.row_stride:] == 0)


def test_feature_embedding_host_surface():
    from rl_ctr_prediction_b200.Feature_embedding import Feature_Embedding
    torch.manual_seed(1)
    port = TP.PortFeatureEmbedding(40, 15, 10)
    torch.manual_seed(1)
    fe = Feature_Embedding(40, 15, 10)
    assert torch.equal(fe.state_dict()["feature_embedding.weight"], port.state_dict()["feature_embedding.weight"])
    assert fe.output_dims == 255 and fe.row[:3] == [0, 0, 0] and fe.col[:3] == [1, 2, 3]
    fe.load_embedding({"feature_embedding.weight": torch.ones(40, 10)})
    assert torch.all(fe.table.data[:, :10] == 1) and torch.all(fe.table.data[:, 10:] == 0)


def test_adam_schedule_matches_torch_scalars():
    from rl_ctr_prediction_b200.tables import AdamSchedule
    s = AdamSchedule(1e-3, (0.9, 0.999), torch.device("cpu"), 16)
    for t in (1, 2, 10, 1500):
        s.ensure(t)
        ss, bc = O.adam_schedule(t, 1e-3)
        assert s.tensor[t, 0].item() == np.float32(ss) and s.tensor[t, 1].item() == np.float32(bc)


def test_models_refuse_cpu_inputs():
    from rl_ctr_prediction_b200 import _lib, p_model
    m = p_model.FM(20, 4)
    with pytest.raises(_lib.RlctrError):
        m(torch.zeros(3, 15, dtype=torch.long))


def test_eva_stopping_and_get_model():
    from rl_ctr_prediction_b200 import pretrain_main as PM
    assert PM.eva_stopping([5, 4, 3, 2, 1], [], "auc") and not PM.eva_stopping([5, 4, 3, 3, 1], [], "auc")
    assert PM.eva_stopping([], [1, 2, 3, 4, 5], "loss") and not PM.eva_stopping([], [1, 2, 3, 4], "loss")
    with pytest.raises(NotImplementedError):
        PM.get_model("nope", 10, 15, 4)


def test_encoded_text_is_parsed_once_and_cached(tmp_path):
    """The CSV of src/encode/data_.py:85 stays the on-disk contract; its int64 image is cached beside it (SURVEY 8f.2)."""
    from rl_ctr_prediction_b200 import pretrain_main as PM
    rng = np.random.default_rng(0)
    rows = np.column_stack([rng.integers(0, 2, 50), rng.integers(0, 1000, (50, 15))]).astype(np.int64)
    path = str(tmp_path / "train.txt")
    np.savetxt(path, rows, delimiter=",", fmt="%d")
    a = PM.load_encoded(path)
    assert np.array_equal(a, rows) and os.path.exists(path + ".int64.npy")
    b = PM.load_encoded(path)                       # second call: memory-mapped image
    assert isinstance(b, np.memmap) and np.array_equal(b, rows)
    rows2 = rows.copy()
    rows2[0, 1] = 7
    np.savetxt(path, rows2, delimiter=",", fmt="%d")
    os.utime(path, (os.path.getmtime(path) + 5, os.path.getmtime(path) + 5))
    assert np.array_equal(PM.load_encoded(path), rows2)      # newer text invalidates the image


def test_agent_memories_refuse_cpu():
    """No CPU fallback anywhere on the product path: the replay memories of the agents live on the device."""
    from rl_ctr_prediction_b200 import _lib, replay, Hybrid_SAC_model
    for cls in (replay.Memory, Hybrid_SAC_model.Memory):
        with pytest.raises(_lib.RlctrError):
            cls(16, 4, "cpu")


def test_td3_action_masking_against_oracle():
    """The rank-comparison form of the TD3 action masking (host torch ops, CPU-checkable) == the oracle's restatement of the
    reference's nonzero loops (v10_Hybrid_TD3_model_PER.py:427-472)."""
    from oracle import np_oracle as O
    from rl_ctr_prediction_b200 import v10_Hybrid_TD3_model_PER as T
    rs = np.random.default_rng(4)
    c = np.tanh(rs.standard_normal((64, 5))).astype(np.float32) * 1.3
    d = rs.random((64, 5)).astype(np.float32)
    eps = rs.standard_normal((64, 5)).astype(np.float32)
    agent = T.Hybrid_TD3_Model.__new__(T.Hybrid_TD3_Model)            # the two helpers use no state
    cur = agent.to_current_state_c_actions(torch.as_tensor(d), torch.as_tensor(c)).numpy()
    nxt = agent.to_next_state_c_actions(torch.as_tensor(d), torch.as_tensor(c), eps=torch.as_tensor(eps)).numpy()
    assert np.array_equal(cur, O.keep_top_d_actions(d, c))
    np.testing.assert_allclose(nxt, O.keep_top_d_actions(d, c, eps), rtol=1e-6, atol=1e-7)


def test_bench_dump_outputs_layout(tmp_path):
    """bench.py --dump-outputs: every model's loss and reference-keyed parameter lands in <name>.npy as float32/float64, the
    N-row tables as the same seeded row sample (so two runs name and index the same values), within the 64 MB cap."""
    import bench
    N = 100_000
    torch.manual_seed(0)
    ms = [(TP.PortCTR(name, N, 15, 10), None) for name in bench.MODELS]
    losses = [torch.tensor([0.5, 0.25, 0.125])]               # a co-located group returns its members' losses as one tensor
    for out in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(out), ms, losses, N)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    total = 0
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), f
        total += a.nbytes
    assert total <= bench.DUMP_MAX_BYTES
    rows = np.load(tmp_path / "a" / "table_rows.npy").astype(np.int64)
    assert len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < N
    for name, (m, _), loss in zip(bench.MODELS, ms, (0.5, 0.25, 0.125)):
        assert np.load(tmp_path / "a" / f"{name}.loss.npy") == np.float32(loss)
        for key, t in m.state_dict().items():
            want = t.numpy()[rows] if t.shape[0] == N else t.numpy()
            assert np.array_equal(np.load(tmp_path / "a" / f"{name}.{key}.npy"), want), (name, key)
