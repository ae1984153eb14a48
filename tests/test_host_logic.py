"""Host-side logic that needs no GPU: metrics vs golden, CLI plumbing (nnet.config, blueprint
loading, bucketing), the extract_embedding chunk rule, world-size-2 sharding under gloo."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from asv_subtools_b200.pipeline import extract_embeddings as cli
from asv_subtools_b200.score import metrics

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _eer_scores(seed):
    rng = np.random.RandomState(seed)
    tar = rng.standard_normal(2000) + 2.0
    non = rng.standard_normal(50000)
    scores = np.concatenate([tar, non])
    labels = np.concatenate([np.ones(2000, dtype=np.int64), np.zeros(50000, dtype=np.int64)])
    perm = rng.permutation(scores.shape[0])
    return scores[perm], labels[perm]


def test_metrics_match_reference_golden(golden):
    g = golden("scoring")
    s, lab = _eer_scores(int(g["eer_scores_seed"]))
    e, t = metrics.eer_bosaris(s, lab)
    assert abs(e - g["eer_bosaris"]) < 1e-12 and abs(t - g["eer_bosaris_thr"]) < 1e-12
    e, t = metrics.eer_det(s, lab)
    assert abs(e - g["eer_det"]) < 1e-12 and abs(t - g["eer_det_thr"]) < 1e-9
    assert abs(metrics.min_dcf(s, lab, 0.01) - g["mindcf_det"]) < 1e-12
    strs = np.where(lab == 1, "target", "nontarget")
    assert metrics.eer_bosaris(s, strs)[0] == metrics.eer_bosaris(s, lab)[0]


def test_metrics_match_oracle_on_ties_and_small_sets():
    from oracle import scoring as osc
    rng = np.random.RandomState(5)
    for n in (40, 400):
        s = np.round(rng.standard_normal(n) + np.repeat([1.0, 0.0], n // 2), 1)  # heavy ties
        lab = np.repeat([1, 0], n // 2)
        assert metrics.eer_bosaris(s, lab) == pytest.approx(osc.eer_bosaris_like(s, lab))
        assert metrics.eer_det(s, lab) == pytest.approx(osc.eer_det_interp(s, lab))
        assert metrics.eer_kaldi(s, lab) == pytest.approx(osc.eer_kaldi(s, lab))


def test_nnet_config_and_blueprint_loading(tmp_path):
    cfg = tmp_path / "nnet.config"
    bp = os.path.join(ROOT, "asv_subtools_b200", "model", "xvector.py")
    # the exact layout pandas.to_csv(header=None, sep=";") writes in utils.write_nnet_config
    cfg.write_text('model_blueprint;{}\nmodel_creation;"Xvector(23,10,training=False,extracted_embedding=""near"")"\n'.format(bp))
    blueprint, creation = cli.read_nnet_config(str(cfg))
    assert blueprint == bp and creation == 'Xvector(23,10,training=False,extracted_embedding="near")'
    m = cli.create_model_from_py(blueprint, creation)
    assert type(m).__name__ == "Xvector" and m.extracted_embedding == "near"
    with pytest.raises(TypeError):
        cli.create_model_from_py(str(tmp_path / "missing.py"), creation)


class FakeModel:
    """Stands in for a blueprint: embedding = [T, mean(feats)] so routing can be checked on CPU."""
    calls = []

    def extract_embedding(self, feats):
        FakeModel.calls.append(("single", feats.shape[0]))
        return torch.tensor([feats.shape[0], float(feats.mean())])

    def extract_embedding_batch(self, x):
        FakeModel.calls.append(("batch", x.shape))
        return torch.stack([torch.tensor([f.shape[0], float(f.mean())]) for f in x])


def test_extract_stream_buckets_by_length_and_shards():
    rng = np.random.RandomState(0)
    lens = [200] * 5 + [300] * 3 + [10001] + [200] * 2
    utts = [("u{}".format(i), rng.standard_normal((t, 4)).astype(np.float32)) for i, t in enumerate(lens)]
    out = {}
    FakeModel.calls = []
    n = cli.extract_stream(FakeModel(), iter(utts), lambda k, v: out.__setitem__(k, v), batch_size=4, log=lambda s: None)
    assert n == len(utts) and set(out) == {k for k, _ in utts}
    for k, f in utts:
        assert out[k][0] == f.shape[0] and abs(out[k][1] - f.mean()) < 1e-6
    kinds = [c[0] for c in FakeModel.calls]
    assert kinds.count("single") == 1                      # only the >maxChunk utterance
    assert ("batch", (4, 200, 4)) in FakeModel.calls       # a full bucket
    out2 = {}
    cli.extract_stream(FakeModel(), iter(utts), lambda k, v: out2.__setitem__(k, v), batch_size=4, shard=(1, 2), log=lambda s: None)
    assert set(out2) == {"u{}".format(i) for i in range(1, len(utts), 2)}
    with pytest.raises(TypeError):
        cli.extract_stream(FakeModel(), iter([("d", np.zeros((3, 4)))]), lambda k, v: None, log=lambda s: None)


def test_chunk_rule_matches_reference_wrapper():
    """for_extract_embedding (framework.py:34-47): the split sizes the plugin base uses."""
    from asv_subtools_b200.nnet.framework import for_extract_embedding

    seen = []

    class M(torch.nn.Module):
        training = False

        def __init__(self):
            super().__init__()
            self.p = torch.nn.Parameter(torch.zeros(1))

        def device_for_extraction(self):
            return torch.device("cpu")

        @for_extract_embedding(maxChunk=100, isMatrix=True)
        def extract_embedding(self, x):
            seen.append(x.shape[1])
            return x.mean(dim=1)

    feats = np.arange(250 * 3, dtype=np.float32).reshape(250, 3)
    e = M().extract_embedding(feats)
    assert seen == [83, 83, 84]                            # num_split=3, split=83, remainder to the last chunk
    assert torch.allclose(e, torch.from_numpy(feats.mean(0)), rtol=1e-6)


@pytest.mark.timeout(120)
def test_world_size_2_gloo_sharding_and_gather(tmp_path):
    """N>1 host logic on CPU: two gloo ranks shard utterances i % 2, all_gather their (fake)
    embeddings and both end with the same, correctly ordered table."""
    script = tmp_path / "w.py"
    script.write_text('''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from asv_subtools_b200.parallel import shard_indices, all_gather_embeddings, all_gather_blocks
dist.init_process_group("gloo")
r, w = dist.get_rank(), dist.get_world_size()
n, d = 11, 4
idx = shard_indices(n, r, w)
local = torch.stack([torch.full((d,), float(i)) for i in idx])
full = all_gather_embeddings(local, n, r, w)
assert full.shape == (n, d) and torch.equal(full[:, 0], torch.arange(n, dtype=torch.float32)), full
# contiguous blocks (the 1 M-utterance job's layout): rank r owns rows [r*5, (r+1)*5)
blk = (torch.arange(5, dtype=torch.float32) + 5 * r)[:, None].repeat(1, d)
tab = all_gather_blocks(blk)
assert tab.shape == (5 * w, d) and torch.equal(tab[:, 0], torch.arange(5 * w, dtype=torch.float32)), tab
print("rank", r, "ok")
dist.destroy_process_group()
''' % ROOT)
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                          "--master-addr", "127.0.0.1", "--master-port", "29617", str(script)],
                         capture_output=True, text=True, timeout=110)
    assert out.returncode == 0, out.stdout + out.stderr
    assert out.stdout.count("ok") == 2


def _run_cli(module, *args):
    return subprocess.run([sys.executable, "-m", module, *args], capture_output=True, text=True, cwd=ROOT,
                          env=dict(os.environ, PYTHONPATH=ROOT), timeout=120)


def test_cli_twins_fail_like_the_reference_clis(tmp_path):
    """Reference contract (SURVEY 8b): on any error the CLIs print a traceback and exit 1 -- the shell wrappers grep
    the logs for it.  Checked here on the paths that fail before any GPU work."""
    r = _run_cli("asv_subtools_b200.score.plda", "only", "three", "args")
    assert r.returncode == 1 and "Traceback" in r.stderr and "expected <trials>" in r.stderr
    r = _run_cli("asv_subtools_b200.score.plda", "--kaldi", "a", "b", "c", "d", "e")
    assert r.returncode == 1 and "num_utts" in r.stderr
    r = _run_cli("asv_subtools_b200.score.compute_plda", str(tmp_path / "missing_spk2utt"), "ark:x", str(tmp_path / "plda"))
    assert r.returncode == 1 and "Traceback" in r.stderr
    r = _run_cli("asv_subtools_b200.score.normalization", "--method", "snorm", "--cross-select", "true",
                 str(tmp_path / "a"), str(tmp_path / "b"), str(tmp_path / "c"), str(tmp_path / "d"))
    assert r.returncode == 1 and "cross-select applies to asnorm" in r.stderr
    r = _run_cli("asv_subtools_b200.pipeline.extract_embeddings", "--use-gpu", "false", "--model-blueprint",
                 os.path.join(ROOT, "asv_subtools_b200", "model", "xvector.py"), "--model-creation",
                 "Xvector(23,10,training=False)", str(tmp_path / "final.params"), "ark:x", "ark:y")
    assert r.returncode == 1 and "no CPU path" in r.stderr
    r = _run_cli("asv_subtools_b200.pipeline.extract_embeddings_online", "--feat-config", str(tmp_path / "missing.yaml"),
                 "--model-blueprint", os.path.join(ROOT, "asv_subtools_b200", "model", "xvector.py"), "--model-creation",
                 "Xvector(80,10,training=False)", str(tmp_path / "final.params"), str(tmp_path / "wav.scp"), "ark:y")
    assert r.returncode == 1 and "Traceback" in r.stderr


def test_blueprints_keep_the_reference_constructor_surface():
    """Creation strings as the launchers write them (runXvector.py:265-266 style) evaluate on every blueprint, expose
    `extracted_embedding`, and carry the reference's state_dict keys."""
    from oracle import nnet as onn
    cases = [("xvector.py", 'Xvector(23,10,training=False,extracted_embedding="far")', onn.xvector_spec(23)),
             ("extended_xvector.py", 'ExtendedXvector(40,10,training=False,extracted_embedding="near")', onn.extended_xvector_spec(40)),
             ("snowdar_xvector.py", 'Xvector(40,10,extend=True,training=False,extracted_embedding="near")', onn.snowdar_xvector_spec(40, extend=True)),
             ("snowdar_xvector.py", 'Xvector(40,10,training=False,pooling="multi-head",pooling_params={"num_head":4,"share":False,'
              '"affine_layers":2})', onn.snowdar_xvector_spec(40, pooling="multi-head",
                                                               pooling_params={"num_head": 4, "share": False, "affine_layers": 2})),
             ("snowdar_xvector.py", 'Xvector(40,10,training=False,pooling="lde",pooling_params={"num_head":12,"num_nodes":200})',
              onn.snowdar_xvector_spec(40, pooling="lde", pooling_params={"num_head": 12, "num_nodes": 200})),
             ("factored_xvector.py", 'Xvector(40,10,training=False,extracted_embedding="far")', onn.factored_xvector_spec(40)),
             ("ecapa_tdnn_xvector.py", 'ECAPA_TDNN(80,10,training=False,extracted_embedding="near",ecapa_params={"channels":1024,'
              '"embd_dim":192,"mfa_conv":1536},fc2_params={"nonlinearity":"","bn":True,"bn_params":{"momentum":0.5,"affine":False,'
              '"track_running_stats":True}})', onn.ecapa_spec(80))]
    for fname, creation, spec in cases:
        m = cli.create_model_from_py(os.path.join(ROOT, "asv_subtools_b200", "model", fname), creation)
        assert hasattr(m, "extracted_embedding") and callable(m.extract_embedding)
        keys = set(m.state_dict().keys())
        want = {e[0] for e in spec}
        assert want <= keys, (fname, sorted(want - keys)[:5])
        extra = {k for k in keys - want if not k.endswith("num_batches_tracked")}
        assert not extra, (fname, sorted(extra)[:5])
        with pytest.raises(RuntimeError):                      # on the CPU: fails loudly, no fallback
            m.extract_embedding(np.zeros((20, m.inputs_dim), dtype=np.float32))


def test_output_pipe_is_waited_for_and_a_failed_command_fails_the_job(tmp_path):
    """ADVICE r1: `ark:| copy-vector ark:- ark,scp:...` must have finished when the writer returns, and a pipe command
    that exits nonzero must raise (the CLIs turn that into exit 1)."""
    import time
    from asv_subtools_b200 import kaldi_io
    out = tmp_path / "v.ark"
    t0 = time.time()
    with kaldi_io.open_or_fd("ark:| sleep 0.5; cat > {}".format(out), "wb") as w:
        kaldi_io.write_vec_flt(w, np.arange(4, dtype=np.float32), key="utt")
    assert time.time() - t0 >= 0.45 and out.exists() and out.stat().st_size > 0
    assert [k for k, _ in kaldi_io.read_vec_flt_ark("ark:cat {} |".format(out))] == ["utt"]
    with pytest.raises(subprocess.CalledProcessError):
        with kaldi_io.open_or_fd("ark:| cat > /dev/null; exit 3", "wb") as w:
            kaldi_io.write_vec_flt(w, np.arange(4, dtype=np.float32), key="utt")


def test_cohort_columns_are_shared_between_score_tables_whatever_their_order():
    """ADVICE r1: AS-norm --cross-select indexes one cohort matrix with the other's top-n columns."""
    from asv_subtools_b200.score import normalization as sn
    keys_a, coh_a = ["e1", "e1", "e1", "e2", "e2", "e2"], ["c1", "c2", "c3", "c1", "c2", "c3"]
    keys_b, coh_b = ["t1", "t1", "t1"], ["c3", "c1", "c2"]
    cidx = sn.cohort_index(coh_a, coh_b)
    ma, _ = sn._dense(keys_a, coh_a, np.arange(6, dtype=np.float32), cidx)
    mb, _ = sn._dense(keys_b, coh_b, np.array([30., 10., 20.], dtype=np.float32), cidx)
    assert cidx == {"c1": 0, "c2": 1, "c3": 2}
    assert mb.tolist() == [[10., 20., 30.]] and ma.tolist() == [[0., 1., 2.], [3., 4., 5.]]
    with pytest.raises(ValueError):   # a table that misses one of the shared columns is incomplete
        sn._dense(["t1", "t1"], ["c1", "c2"], np.zeros(2, dtype=np.float32), cidx)


def test_batcher_buckets_by_a_length_key_and_flushes_incrementally():
    """ADVICE r1: the waveform CLI buckets by frame count with a finite amount held back."""
    b = cli.Batcher(2, max_pending_frames=10, length=lambda w: w.shape[0] // 4)
    out = []
    for i, n in enumerate([8, 9, 16, 17, 4, 24, 32]):
        out += [[k for k, _ in bucket] for bucket in b.add("u%d" % i, np.zeros(n, dtype=np.float32))]
    out += [[k for k, _ in bucket] for bucket in b.flush()]
    assert out[0] == ["u0", "u1"] and out[1] == ["u2", "u3"]          # equal FRAME counts share a bucket
    assert sorted(k for bucket in out for k in bucket) == ["u%d" % i for i in range(7)]
    assert len(out) >= 4                                               # the pending cap flushed before the end


def test_host_side_plda_interpolators_match_reference_golden(golden, tmp_path):
    """LIP / LIP-reg are pure float64 host algebra (no adaptation vectors, no Gram product): checked here on the CPU
    against the reference's own classes; the CORAL-based members of the family are GPU tests."""
    from asv_subtools_b200 import kaldi_io
    from asv_subtools_b200.score.plda_train import Lip, LipReg, _excess_over
    from oracle import plda_train as opt
    g, ga = golden("plda_train"), golden("plda_adapt")
    paths = []
    for name, (m, w, b) in (("out", (g["d16_mean"], g["d16_within"], g["d16_between"])),
                            ("in", (ga["in_mean"], ga["in_within"], ga["in_between"]))):
        p = str(tmp_path / (name + ".ori"))
        with open(p, "wb") as f:
            kaldi_io.write_vec_flt(f, m.reshape(-1), key="mean")
            kaldi_io.write_vec_flt(f, w.reshape(-1), key="within_var")
            kaldi_io.write_vec_flt(f, b.reshape(-1), key="between_var")
        paths.append(p)
    for key, cls in (("lip", Lip), ("lipreg", LipReg)):
        m = cls()
        m.interpolation(*paths)
        for got, want in ((m.mean.reshape(-1), ga[key + "_mean"]), (m.within_var, ga[key + "_within"]), (m.between_var, ga[key + "_between"])):
            assert np.max(np.abs(got - want)) / np.max(np.abs(want)) < 1e-9, key
    x = _excess_over(ga["in_within"], g["d16_within"])
    assert np.max(np.abs(x - opt.covariance_regulariser(ga["in_within"], g["d16_within"]))) < 1e-10 * np.max(np.abs(x))
    assert np.min(np.linalg.eigvalsh(x)) > -1e-10            # a positive semi-definite excess


def test_backend_transform_host_algebra_matches_oracle_and_reference(golden):
    """The D x D float64 halves of trainlda / trainwhiten / trainpcawhiten (score/process.py) on statistics computed
    in NumPy: ZCA against the reference script's matrix, LDA / PCA against the oracle (sign-free comparisons)."""
    from asv_subtools_b200.score import process as proc
    from oracle import scoring as osc
    g = golden("whiten")
    x = g["emb"].astype(np.float64)
    assert np.max(np.abs(proc.zca_from_gram(x.T @ x, x.shape[0]) - g["zca"])) < 1e-6
    emb, lab = osc.synthetic_speakers(40, 6, 16, 5, noise=0.9)
    emb = emb.astype(np.float64) + 0.7
    mean = emb.mean(0)
    xc = emb - mean
    total = xc.T @ xc / emb.shape[0]
    means = np.stack([xc[lab == s].mean(0) for s in np.unique(lab)])
    between = (means.T * np.bincount(lab)) @ means / emb.shape[0]
    got, want = proc.lda_from_statistics(mean, total, between, 6), osc.lda_transform(emb, lab, 6)
    sign = np.sign(np.sum(got[:, :16] * want[:, :16], axis=1))[:, None]
    assert np.max(np.abs(got * sign - want)) < 1e-8
    got, want = proc.pca_from_statistics(mean, total), osc.pca_transform(emb)
    sign = np.sign(np.sum(got[:, :16] * want[:, :16], axis=1))[:, None]
    assert np.max(np.abs(got * sign - want)) < 1e-8


def test_bench_shard_balancing_keeps_the_total_and_whole_batches():
    """bench.balance_shards: sizes follow the measured speeds in whole batches, the total is exact, the odd tail goes to the
    fastest rank, and an impossible cut (over the per-rank capacity) is refused rather than approximated."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n, B = 125000, 256
    cap = n + ((n * 8 // 100 + B - 1) // B) * B
    for speed in ([1.0, 1.0], [1.0, 0.96], [1, 0.97, 1.02, 0.99, 1.0, 0.95, 1.03, 1.0]):
        cut = bench.balance_shards(speed, n * len(speed), B, cap)
        assert cut is not None and sum(cut) == n * len(speed) and max(cut) <= cap
        fastest = int(np.argmax(speed))
        assert all(c % B == 0 for i, c in enumerate(cut) if i != fastest)
        order = np.argsort(speed)
        assert all(cut[order[i]] <= cut[order[i + 1]] + B for i in range(len(speed) - 1))      # monotone in speed up to one batch
    assert bench.balance_shards([1.0, 0.5], 2 * n, B, cap) is None                               # would need 167 k on one rank
    assert bench.balance_shards([1.0, 1.0], 2 * n, B, cap) == [125072, 124928]


def test_bench_dump_outputs_writes_a_fixed_float32_sample_of_rows(tmp_path):
    """bench.dump_outputs (--dump-outputs): float32 .npy files under 64 MB; a table longer than DUMP_ROWS is cut to the same
    rows on every call, taken unchanged; a short one is written whole."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    n = bench.DUMP_ROWS + 5000
    table = torch.arange(n, dtype=torch.float64)[:, None].repeat(1, 512)      # row i holds i
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), embeddings=table, short=table[:100])
    a, b = np.load(tmp_path / "a" / "embeddings.npy"), np.load(tmp_path / "b" / "embeddings.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_ROWS, 512) and np.array_equal(a, b)
    rows = a[:, 0]
    assert np.all(a == rows[:, None]) and np.all(np.diff(rows) > 0) and rows[-1] < n
    assert np.array_equal(np.load(tmp_path / "a" / "short.npy"), table[:100].float().numpy())
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 << 20


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (the CPU arm the driver runs beside the native one): one JSON line with the contract's keys,
    `impl` = reference, the same metric / unit / config keys as the native arm, an `e2e` block without copies, no GPU needed;
    and without a GPU the native arm refuses to run instead of falling back."""
    import json
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3"],
                       capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches", "impl"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["config"]["batch"] == 256 and line["config"]["frames_per_utt"] == 200 and "workload" in line["config"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["value"] > 0
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0 and line["gpu_launches"] == 0
    if not torch.cuda.is_available():
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, env=env, cwd=ROOT,
                           timeout=300)
        assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
