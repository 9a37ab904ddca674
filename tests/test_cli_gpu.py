"""GPU: the drop-in command lines end to end on small image folders written to disk, against the oracle pipeline
(dataset order -> transform -> SSCD forward -> normalise -> mm -> topk -> statistics)."""
import json
import os
import pickle as pkl

import numpy as np
import pytest
import torch

from dcr_b200 import cli, data, embedding_search as es
from oracle import models as om
from oracle import similarity as osim

pytestmark = pytest.mark.gpu


def _write_images(folder, n, seed, names=None):
    from PIL import Image
    os.makedirs(folder, exist_ok=True)
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (n, 8, 8, 3), dtype=np.uint8)
    imgs = np.stack([np.asarray(Image.fromarray(b).resize((256, 256), Image.BILINEAR)) for b in base])
    imgs = np.clip(imgs.astype(np.int16) + rng.integers(-20, 21, imgs.shape), 0, 255).astype(np.uint8)
    for i in range(n):
        Image.fromarray(imgs[i]).save(os.path.join(folder, names[i] if names else f"{i}.png"))
    with open(os.path.join(folder, "prompts.txt"), "w") as f:
        f.writelines(f"prompt {i}\n" for i in range(n))
    return imgs


def test_diff_retrieval_cli_end_to_end(tmp_path, monkeypatch, capsys):
    monkeypatch.chdir(tmp_path)
    q_dir, v_dir = str(tmp_path / "runs" / "exp" / "generations"), str(tmp_path / "train")
    q_imgs = _write_images(q_dir, 12, 1)
    v_imgs = _write_images(v_dir, 30, 2)
    # three near-copies of training images among the generations
    from PIL import Image
    for j, src in enumerate([3, 11, 25]):
        Image.fromarray(v_imgs[src]).save(os.path.join(q_dir, f"{j}.png"))
        q_imgs[j] = v_imgs[src]
    sd = om.make_sscd_state_dict(7)
    wpath = str(tmp_path / "sscd.pt")
    torch.save(sd, wpath)
    rc = cli.main(["--query_dir", q_dir, "--val_dir", v_dir, "--pt_style", "sscd", "--arch", "resnet50",
                   "--similarity_metric", "dotproduct", "--weights", wpath, "--precision", "exact", "--topk", "5"])
    assert rc == 0
    save = os.path.join("ret_plots", "runs", "exp", "generations", "images", "sscd_resnet50_dotproduct")   # :378,:408
    res = torch.load(os.path.join(save, "topk.pth"))
    stats = json.load(open(os.path.join(save, "stats.json")))
    # oracle pipeline on the same files in SynthDataset order (natsorted paths)
    qf, vf = data.list_images(q_dir), data.list_images(v_dir)
    assert [os.path.basename(f) for f in qf] == [f"{i}.png" for i in range(12)]
    assert res["query_files"] == qf and res["gallery_files"] == vf
    qd = om.sscd_forward(sd, om.preprocess(torch.from_numpy(q_imgs))).numpy()
    vd = om.sscd_forward(sd, om.preprocess(torch.from_numpy(v_imgs))).numpy()
    qd, vd = osim.l2_normalize(qd), osim.l2_normalize(vd)
    ov, oi = osim.sim_topk(qd, vd, 5)
    got_i, got_v = res["indices"].numpy(), res["values"].numpy()
    assert np.array_equal(got_i[:, 0], oi[:, 0])                      # best match per generation
    assert got_i[:3, 0].tolist() == [3, 11, 25] and np.all(got_v[:3, 0] > 0.9999)
    np.testing.assert_allclose(got_v, ov, atol=1e-4)                  # north-star tolerance on scores
    ref_stats = osim.retrieval_stats(ov[:, 0], osim.background_second_best(vd))
    for k, v in ref_stats.items():
        assert abs(stats[k] - v) < 1e-4, (k, stats[k], v)
    assert "Simscores @x% part done" in capsys.readouterr().out          # diff_retrieval.py:470


def test_embedding_search_cli_end_to_end(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    sd = om.make_sscd_state_dict(8)
    wpath = str(tmp_path / "sscd.pt")
    torch.save(sd, wpath)
    laion = tmp_path / "laion"
    all_imgs = {}
    for part, (n, seed) in {"part_a": (9, 3), "part_b": (7, 4)}.items():
        folder = str(tmp_path / "raw" / part)
        names = [f"img{i:03d}.png" for i in range(n)]
        all_imgs[part] = (_write_images(folder, n, seed, names), names)
        os.remove(os.path.join(folder, "prompts.txt"))
        assert es.embed_main(["--image-folder", folder, "--dump-path", str(laion / part), "--weights", wpath,
                              "--batch-size", "4", "--workers", "1"]) == 0
    gen_folder = str(tmp_path / "raw" / "gen")
    gen_names = ["g1.png", "g0.png", "g2.png"]
    gen_imgs = _write_images(gen_folder, 3, 5, gen_names)
    from PIL import Image
    Image.fromarray(all_imgs["part_b"][0][4]).save(os.path.join(gen_folder, "g0.png"))     # a copy of part_b/img004
    es.embed_main(["--image-folder", gen_folder, "--dump-path", str(tmp_path / "gen_emb"), "--weights", wpath, "--workers", "1"])
    out_path = str(tmp_path / "result.pkl")
    assert es.search_main(["--laion-embedding-folder", str(laion), "--generation-embedding-path",
                           str(tmp_path / "gen_emb" / "embedding.pkl"), "--dump-path", out_path]) == 0
    with open(out_path, "rb") as f:
        out = pkl.load(f)
    assert out["gen_images"] == ["g0.png", "g1.png", "g2.png"]           # sorted file names (utils.py:123)
    assert out["keys"][0] == "part_b:img004.png" and out["scores"][0] > 0.9999
    from oracle import embedding_search as oes
    ref = oes.similarity_search(str(laion), str(tmp_path / "gen_emb" / "embedding.pkl"))
    assert out["keys"].tolist() == ref["keys"].tolist()
    np.testing.assert_allclose(out["scores"], ref["scores"], atol=1e-6)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_diff_retrieval_cli_multiprocessing_distributed(tmp_path, monkeypatch):
    """`--multiprocessing-distributed --world-size 1 --rank 0 --dist-url tcp://...` (diff_retrieval.py:205-246): one worker
    per GPU, gallery and queries sharded, per-shard top-k merged over NCCL -- same topk.pth and statistics as the
    single-process run of the same command."""
    import subprocess
    import sys
    monkeypatch.chdir(tmp_path)
    q_dir, v_dir = str(tmp_path / "runs" / "exp" / "generations"), str(tmp_path / "train")
    _write_images(q_dir, 11, 21)
    _write_images(v_dir, 37, 22)
    sd = om.make_sscd_state_dict(7)
    wpath = str(tmp_path / "sscd.pt")
    torch.save(sd, wpath)
    common = ["--query_dir", q_dir, "--val_dir", v_dir, "--pt_style", "sscd", "--arch", "resnet50", "--weights", wpath,
              "--precision", "parity", "--topk", "5"]
    save = os.path.join("ret_plots", "runs", "exp", "generations", "images", "sscd_resnet50_dotproduct")
    assert cli.main(common) == 0
    single = torch.load(os.path.join(save, "topk.pth"))
    single_stats = json.load(open(os.path.join(save, "stats.json")))
    os.remove(os.path.join(save, "topk.pth"))
    port = 29500 + os.getpid() % 1000
    env = dict(os.environ, PYTHONPATH=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    r = subprocess.run([sys.executable, "-m", "dcr_b200.cli", *common, "--multiprocessing-distributed", "--world-size", "1",
                        "--rank", "0", "--dist-url", f"tcp://127.0.0.1:{port}"], env=env, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    multi = torch.load(os.path.join(save, "topk.pth"))
    assert torch.equal(multi["indices"], single["indices"])
    assert torch.allclose(multi["values"], single["values"], atol=1e-6)
    stats = json.load(open(os.path.join(save, "stats.json")))
    for k, v in single_stats.items():
        assert abs(stats[k] - v) < 1e-6, (k, stats[k], v)
