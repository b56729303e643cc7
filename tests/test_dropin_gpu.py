"""The drop-in, proven through the reference's OWN entry point on a GPU: the unmodified
`MuseDiffusion.run.sample.main()` (run/sample.py:22-311, from the verbatim copy oracle/_ref/ that oracle/build_ref.sh makes)
is run twice on the same reference-written checkpoint directory (`model_000000.pt` + `TrainSettings(...).json()`), the same
inputs and the same noise stream — once with its stock modules on the host CPU, once with the three `sys.modules`
swaps of INTEGRATION.md so that `create_model_and_diffusion`, the loops and the rounding callback resolve to
musediffusion_b200 on cuda:0.  Tokens handed to `decode_batch` must be the reference's under the north-star rule
(oracle/parity_rule.py): ids equal at every rounding call except below-margin positions.

Those three tests need the reference's source, which the repository does not hold.  The `test_package_main_*` tests below
run without it: the package's own port of that entry point (`musediffusion_b200.sample.main`) with the same arguments, a
model directory holding the reference-written training_args.json of tests/golden, the same noise stream and the same rule,
against the numpy oracle (itself pinned to the reference's fixtures by test_oracle_golden.py).  They cover the driver
around the loops: --step -> DDPM or DDIM gap, --strength -> noising_t and the q_sample at noising_t - 1, the generation-mode
meta prefix and masking, two batches drawn from one noise stream, the tokens handed to decode_batch and the MIDI files."""
import json
import os

import numpy as np
import pytest
import torch

import musediff_oracle as O
import parity_rule as R
import ref_harness as H

pytestmark = pytest.mark.gpu
if not torch.cuda.is_available():  # pragma: no cover
    pytest.skip("needs a CUDA device", allow_module_level=True)
needs_reference = pytest.mark.skipif(
    not H.available(), reason="needs the unmodified MuseDiffusion source tree (oracle/_ref/ or $MUSEDIFFUSION_REFERENCE), "
                              "which is not part of the repository")

MARGIN_TOL, DOWNSTREAM_TOL = 0.5, 1.0
L = 64
META = ["--bpm", "70", "--audio_key", "aminor", "--time_signature", "4/4", "--pitch_range", "mid_high", "--num_measures", "8",
        "--inst", "acoustic_piano", "--genre", "newage", "--min_velocity", "60", "--max_velocity", "80", "--track_role",
        "main_melody", "--rhythm", "standard", "--chord_progression", "Am-Am-Am-Am-G-G-G-G-F-F-F-F-E-E-E-E"]


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    d = tmp_path_factory.mktemp("dropin")
    H.install()
    p = O.make_random_params(seed=7, seq_len=L)
    return H.write_checkpoint_dir(str(d / "diffusion_models"), p, seq_len=L), str(d / "out")


def compare(tag, ref, got):
    assert len(ref["tokens"]) == len(got["tokens"]) >= 1
    n_batches = len(ref["tokens"])
    calls = len(ref["step_ids"]) // n_batches
    assert len(got["step_ids"]) == len(ref["step_ids"]) and calls >= 1
    for b in range(n_batches):
        rt, gt, mask = ref["tokens"][b], got["tokens"][b], ref["masks"][b]
        assert gt.dtype == rt.dtype and gt.shape == rt.shape and np.array_equal(got["masks"][b], mask)
        ref_ids = np.stack(ref["step_ids"][b * calls:(b + 1) * calls])
        ref_margin = np.stack(ref["step_margin"][b * calls:(b + 1) * calls])
        got_ids = np.stack(got["step_ids"][b * calls:(b + 1) * calls])
        free = mask != 0
        rep = R.chain_report(ref_ids, ref_margin, got_ids, free, MARGIN_TOL, DOWNSTREAM_TOL)
        tk = R.token_report(rt, gt, free, rep["never_divergent"])
        print("%s batch %d: %d rounding calls, ids equal at %.5f of (call, position) pairs, %d below-margin positions "
              "(max margin %.3f), tokens equal at %.5f; violations %d + %d"
              % (tag, b, calls, rep["id_agreement_all_calls"], rep["positions_ever_divergent"],
                 max(rep["max_margin_primary"], rep["max_margin_downstream"]), tk["token_agreement"], rep["violations"],
                 tk["token_violations"]))
        assert rep["violations"] == 0 and tk["token_violations"] == 0, (rep, tk)
        assert np.array_equal(gt[~free & (rt > 0)], rt[~free & (rt > 0)])        # the conditioning prefix comes back untouched


@needs_reference
def test_reference_main_generation_dropin(checkpoint):
    model_path, out_dir = checkpoint
    argv = ["--step", "20", "--batch_size", "2", "--num_samples", "2"] + META          # DDIM, gap 100
    ref = H.run_main("generation", model_path, out_dir, argv, stream_seed=5)
    got = H.run_main("generation", model_path, out_dir, argv, dropin=True, stream_seed=5)
    compare("generation / ddim20", ref, got)


@needs_reference
def test_reference_main_modification_dropin(checkpoint):
    model_path, out_dir = checkpoint
    conds = [O.make_synthetic_batch("modification", 3, L, seed=3 + i) for i in range(2)]
    batches = [{k: torch.from_numpy(v) for k, v in c.items()} for c in conds]
    argv = ["--step", "2000", "--batch_size", "3", "--strength", "0.006", "--use_corruption", "false"]   # DDPM, t_enc = 12, top_p = 1
    ref = H.run_main("modification", model_path, out_dir, argv, batches=batches, stream_seed=6)
    got = H.run_main("modification", model_path, out_dir, argv, batches=batches, dropin=True, stream_seed=6)
    compare("modification / ddpm x12", ref, got)
    argv = ["--step", "50", "--batch_size", "3", "--strength", "0.5", "--use_corruption", "false"]       # DDIM gap 40, t_enc = 25
    ref = H.run_main("modification", model_path, out_dir, argv, batches=batches, stream_seed=8)
    got = H.run_main("modification", model_path, out_dir, argv, batches=batches, dropin=True, stream_seed=8)
    compare("modification / ddim50 x25", ref, got)


@needs_reference
def test_reference_main_ends_in_midi_files(checkpoint, capsys):
    """fourth swap: `decode_batch` of the reference's main() resolves to the package's (GPU validity filter + MIDI writer);
    the run's own bookkeeping (valid counts, log file) goes on as with the reference's decoder."""
    model_path, out_dir = checkpoint
    conds = [O.make_synthetic_batch("modification", 3, L, seed=30 + i) for i in range(2)]
    batches = [{k: torch.from_numpy(v) for k, v in c.items()} for c in conds]
    argv = ["--step", "20", "--batch_size", "3", "--strength", "0.5", "--use_corruption", "false"]
    got = H.run_main("modification", model_path, out_dir, argv, batches=batches, dropin=True, stream_seed=9, midi_tail=True)
    assert len(got["valid"]) == 2
    files = sorted(f for f in os.listdir(got["output_dir"]) if f.endswith(".midi"))
    want = []
    for b, (count, invalid) in enumerate(got["valid"]):
        assert count + len(invalid) == 3
        want += ["%07d_batch%05d_%04d.midi" % (b * 3 + k, b, k) for k in range(3) if k not in invalid]
    assert files == sorted(want)
    printed = capsys.readouterr().out
    assert printed.count("Summary of Batch") >= 2


# ------------------------------------------------------------------------------------ without the reference's source
@pytest.fixture(scope="module")
def package_model(tmp_path_factory, golden_dir):
    """a model directory as the reference's trainer leaves it: its training_args.json (tests/golden, at L = 64, corruption
    off) next to `model_000000.pt`; the weights of the drop-in tests above."""
    d = tmp_path_factory.mktemp("main") / "diffusion_models"
    d.mkdir()
    raw = json.load(open(os.path.join(golden_dir, "training_args_default.json")))
    raw.update(seq_len=L, use_corruption=False)
    (d / "training_args.json").write_text(json.dumps(raw))
    p = O.make_random_params(seed=7, seq_len=L)
    torch.save({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in p.items()}, str(d / "model_000000.pt"))
    return str(d / "model_000000.pt"), p


def run_package_main(mode, model_path, out_dir, argv, stream_seed):
    """musediffusion_b200.sample.main with the oracle's noise stream injected and every rounding call traced; returns the
    run's dict in the layout of `H.run_main` (the tokens per batch are what main() hands to decode_batch)."""
    import musediffusion_b200.diffusion as D
    from musediffusion_b200.sample import main
    stream = O.NoiseStream(stream_seed)
    D.GaussianDiffusion.noise_source = staticmethod(
        lambda shape, kind: stream.truncated(shape, 1) if kind == "truncated" else stream.randn(shape))
    trace = []
    D.GaussianDiffusion.rounding_trace = trace
    try:
        main([mode, "--model_path", model_path, "--out_dir", out_dir] + list(argv))
    finally:
        D.GaussianDiffusion.noise_source = None
        D.GaussianDiffusion.rounding_trace = None
    out = os.path.join(out_dir, "diffusion_models", os.path.basename(model_path) + "." + mode + ".samples")
    batch = int(argv[argv.index("--batch_size") + 1])
    tokens = np.load(os.path.join(out, "tokens.npy"))
    got = {"tokens": [tokens[k:k + batch] for k in range(0, len(tokens), batch)], "output_dir": out,
           "status": np.load(os.path.join(out, "decode_status.npy"))}
    got["step_ids"] = [ids.view(-1, L).cpu().numpy() for ids, _ in trace]
    got["step_margin"] = [m.view(-1, L).cpu().numpy() for _, m in trace]
    return got


def run_oracle(p, batches, mode, step, strength, stream_seed):
    """run/sample.py:177-220 per batch in the numpy oracle, the batches in order from one noise stream."""
    s = O.make_schedule("sqrt", 2000)
    stream = O.NoiseStream(stream_seed)
    ref = {"tokens": [], "masks": [], "step_ids": [], "step_margin": []}
    for cond in batches:
        record = []
        ref["tokens"].append(O.sample_batch(s, p, cond, mode, step, stream, strength=strength, top_p=1, record=record))
        ref["masks"].append(np.asarray(cond["input_mask"]))
        ids, margin = R.oracle_chain_trace(record, p["word_embedding.weight"])
        ref["step_ids"] += list(ids)
        ref["step_margin"] += list(margin)
    return ref


def modification_batches(tmp_path, seeds, B=3):
    conds = [O.make_synthetic_batch("modification", B, L, seed=s) for s in seeds]
    for c in conds:
        # main() writes MIDI files, which cannot carry an "unknown" tempo / key / time signature (the reference's writer raises
        # on them too): the first known class instead, as main() does for its own synthetic input
        for col, unknown in ((0, 560), (1, 601), (2, 626)):
            c["input_ids"][:, col] = np.where(c["input_ids"][:, col] == unknown, unknown + 1, c["input_ids"][:, col])
    path = str(tmp_path / "batches.npz")
    np.savez(path, input_ids=np.concatenate([c["input_ids"] for c in conds]),
             input_mask=np.concatenate([c["input_mask"] for c in conds]))
    return conds, path


def test_package_main_generation(package_model, tmp_path):
    from musediffusion_b200.meta import meta_from_args, meta_to_batch
    from musediffusion_b200.sample import create_parser
    model_path, p = package_model
    argv = ["--step", "20", "--batch_size", "2", "--num_samples", "2"] + META          # DDIM, gap 100
    b = meta_to_batch(meta_from_args(create_parser().parse_args(["generation", "--model_path", model_path] + argv)), 2, L)
    cond = {"input_ids": b["input_ids"].numpy(), "input_mask": b["input_mask"].numpy()}
    got = run_package_main("generation", model_path, str(tmp_path / "out"), argv, stream_seed=5)
    got["masks"] = [cond["input_mask"]]
    compare("package main, generation / ddim20", run_oracle(p, [cond], "generation", 20, 1.0, 5), got)


def test_package_main_modification(package_model, tmp_path):
    model_path, p = package_model
    conds, npz = modification_batches(tmp_path, (3, 4))
    for argv, step, strength, seed in ((["--step", "2000", "--strength", "0.006"], 2000, 0.006, 6),    # DDPM, t_enc = 12
                                       (["--step", "50", "--strength", "0.5"], 50, 0.5, 8)):           # DDIM gap 40, t_enc = 25
        argv = argv + ["--batch_size", "3", "--num_batches", "2", "--input_npz", npz, "--use_corruption", "false"]
        got = run_package_main("modification", model_path, str(tmp_path / ("out%d" % seed)), argv, stream_seed=seed)
        got["masks"] = [c["input_mask"] for c in conds]
        compare("package main, modification / step %d x %d" % (step, int(step * strength)),
                run_oracle(p, conds, "modification", step, strength, seed), got)


def test_package_main_ends_in_midi_files(package_model, tmp_path, capsys):
    """main()'s decode_batch tail: one MIDI file per valid row, named and numbered as the reference's writer does."""
    from musediffusion_b200 import decode_util
    model_path, _ = package_model
    _, npz = modification_batches(tmp_path, (30, 31))
    argv = ["--step", "20", "--batch_size", "3", "--num_batches", "2", "--strength", "0.5", "--input_npz", npz,
            "--use_corruption", "false"]
    got = run_package_main("modification", model_path, str(tmp_path / "out"), argv, stream_seed=9)
    files = sorted(f for f in os.listdir(got["output_dir"]) if f.endswith(".midi"))
    ok = got["status"] == decode_util.OK
    assert ok.shape == (6,)
    assert files == sorted("%07d_batch%05d_%04d.midi" % (n, n // 3, n % 3) for n in np.nonzero(ok)[0])
    assert capsys.readouterr().out.count("Summary of Batch") >= 2
