"""Epoch loops of the drivers with the host overheads removed (SURVEY.md 8(f) row f3).

`train` and `evaluate` keep the signatures and return values of main.py:54-96 and :98-180.  What changes is
where the per-batch bookkeeping happens: the reference synchronises three times per batch for the running
totals (main.py:83-85), copies the [B,N,3] reconstruction to the host and runs the de-normalisation, the
Procrustes back-transform (`bmm`) and the vertex errors there (main.py:88-94).  Here every batch ends with two
launches on the device - `mvb_recon_error` on the decoder's buffer and `mvb_epoch_meter_add` into eight fp64
accumulators - and the epoch ends with ONE read-back.  `train_epoch` is the same loop on the captured
`engine.TrainEngine` step (fixed batch size replayed as a CUDA graph; the ragged last batch runs uncaptured).

`inference` is the batch loop of `inference.py` (:55-157) with the same three report files and OBJ outputs.
`estimate_diff`, `train_classifier` and `evaluate_classifier` are the counterparts for `crecon.py` (:64-150, :162-201):
the sex classifier `cheb_GCN` trained on the residuals of the VAE's reconstruction under both labels.
"""
import os

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import dp, formats
from . import functional as Fn


def _split(data):
    x, x_gt, y, names, gt_mesh, R, m, s = data
    return x, x_gt, y, names, gt_mesh, R, m, s


def _norm(checkpoint_dir, norm, device):
    mean, std = norm if norm is not None else formats.load_norm(checkpoint_dir)
    return (torch.as_tensor(mean, dtype=torch.float32).to(device), torch.as_tensor(std, dtype=torch.float32).to(device))


def _num_graphs(x):
    return x.shape[0] if torch.is_tensor(x) else x.num_graphs


def train(model, train_loader, optimizer, device, checkpoint_dir=None, norm=None):
    """main.py:54-96.  -> (loss, kld, rec_loss, error, accuracy) per-sample means over the epoch (numpy float64
    scalars: `.item()` works on each, as the driver expects of the accuracy).  `norm` = (mean, std) replaces the
    norm.npz read."""
    model.train()
    mean, std = _norm(checkpoint_dir, norm, device)
    meter = Fn.EpochMeter(device)
    for data in train_loader:
        x, x_gt, y, _, gt_mesh, R, m, s = _split(data)
        x, x_gt = x.to(device, non_blocking=True), x_gt.to(device, non_blocking=True)
        sex_hot = F.one_hot(y, num_classes=2).to(device, non_blocking=True)
        optimizer.zero_grad()
        loss, correct, out, z, _ = model(x, x_gt, sex_hot, m_type="train")
        loss.backward()
        optimizer.step()
        mean_err, _ = Fn.recon_error(out.detach(), mean, std, s, R, m, gt_mesh)
        meter.add(loss, z[0], z[1], correct, mean_err)
    r = meter.read()
    return r["loss"], r["kld"], r["rec_loss"], r["error"], np.float64(r["accuracy"])


def train_epoch(engine, train_loader, checkpoint_dir=None, norm=None):
    """`train` on the captured step with the input double-buffered: while step i computes, batch i+1 is already on
    its way to the device (`engine.stage` / `engine.step_prefetched`, nothing read back per batch);
    `engine.ragged_step` for a smaller last batch.  Same return tuple."""
    dev = engine.dev
    engine.net.train()
    mean, std = _norm(checkpoint_dir, norm, dev)
    meter = Fn.EpochMeter(dev)

    def host_batch(data):
        x, x_gt, y = data[0], data[1], data[2]
        b = _num_graphs(x)
        xt = (x if torch.is_tensor(x) else x.x).reshape(b, engine.n_vert, engine.feat)
        return b, (xt, x_gt.reshape(b, engine.n_vert, engine.feat), y)

    # Which path a step takes - the replayed graphs (bucketed all-reduces) or the uncaptured ragged step (one
    # all-reduce) - must be the SAME on every rank: it is decided from the size of the GLOBAL batch (a loader that
    # knows it: ShardedMeshLoader.global_chunk_sizes), else by agreement (a MIN all-reduce of "my slice is full").
    world, rank = engine.world, (dist.get_rank() if engine.world > 1 else 0)
    sizes = train_loader.global_chunk_sizes() if hasattr(train_loader, "global_chunk_sizes") else None

    def full_everywhere(i, b):
        if world == 1:
            return b == engine.batch, 1.0
        if sizes is not None:
            g = sizes[i]
            return g == engine.batch * world, dp.ragged_weight(g, rank, world)
        flag = torch.tensor([1 if b == engine.batch else 0, b], device=dev, dtype=torch.int64)
        both = [torch.zeros_like(flag) for _ in range(world)]
        dist.all_gather(both, flag)
        g = int(sum(int(t[1]) for t in both))
        return all(int(t[0]) for t in both), b * world / float(max(g, 1))

    it = iter(train_loader)
    cur = next(it, None)
    staged = False
    i = 0
    cur_full = full_everywhere(0, host_batch(cur)[0]) if cur is not None else (False, 1.0)
    while cur is not None:
        nxt = next(it, None)
        b, hb = host_batch(cur)
        nxt_full = full_everywhere(i + 1, host_batch(nxt)[0]) if nxt is not None else (False, 1.0)
        _, _, _, _, gt_mesh, R, m, s = _split(cur)
        if cur_full[0]:
            if not staged:
                engine.stage(*hb)
            staged = nxt is not None and nxt_full[0]
            engine.step_prefetched(host_batch(nxt)[1] if staged else None, sync=False)
            loss, kld, rec, correct, recon = engine.loss, engine.kld, engine.rec, engine.correct, engine.recon
        else:
            xt, x_gt, y = hb
            y_hot = F.one_hot(y, num_classes=engine.net.num_class).to(dev)
            loss, kld, rec, correct, recon = engine.ragged_step(xt.to(dev), x_gt.to(dev, engine.x_gt.dtype), y_hot,
                                                                grad_weight=cur_full[1])
            staged = False
        i += 1
        cur_full = nxt_full
        mean_err, _ = Fn.recon_error(recon, mean, std, s, R, m, gt_mesh)
        meter.add(loss, kld, rec, correct, mean_err)
        cur = nxt
    r = meter.read()
    return r["loss"], r["kld"], r["rec_loss"], r["error"], np.float64(r["accuracy"])


def classifier_(net, x):
    """main.py:42-49: predicted class of a batch of (normalised) meshes"""
    return torch.argmax(net.classifier(net.encoder(x)), dim=1)


def evaluate(n, model, test_loader, device, faces=None, checkpoint_dir=None, vis=False, norm=None):
    """main.py:98-180.  -> (loss, kld, rec_loss, accuracy, errors [n_meshes, N] per-vertex distances, sex-change
    success rate).  Per batch: forward, the sex-changed decode + re-classification (main.py:153-160), error kernel,
    meter; nothing is read back before the end of the loop unless vis=True (OBJ files need the meshes)."""
    model.eval()
    mean, std = _norm(checkpoint_dir, norm, device)
    meter = Fn.EpochMeter(device)
    flipped = torch.zeros((), device=device, dtype=torch.int64)
    errors = []
    ok_dir = bad_dir = None
    if vis:
        save_path = os.path.join(checkpoint_dir, "mesh" + str(n))
        ok_dir, bad_dir = os.path.join(save_path, "sex_change_S"), os.path.join(save_path, "sex_change_F")
        os.makedirs(ok_dir, exist_ok=True)
        os.makedirs(bad_dir, exist_ok=True)
    with torch.no_grad():
        for data in test_loader:
            x, x_gt, y, names, gt_mesh, R, m, s = _split(data)
            x, x_gt = x.to(device, non_blocking=True), x_gt.to(device, non_blocking=True)
            sex_hot = F.one_hot(y, num_classes=2).to(device, non_blocking=True)
            loss, correct, out, z, _ = model(x, x_gt, sex_hot, m_type="test")
            res = Fn.recon_error(out, mean, std, s, R, m, gt_mesh, per_vertex=True, mesh=vis)
            meter.add(loss, z[0], z[1], correct, res[0])
            errors.append(res[2])
            oppo = 1 - sex_hot
            index_gt = torch.argmax(oppo, dim=1)
            oppo_x = model.sample(oppo, z[2])
            index_pred = classifier_(model, oppo_x)
            flipped += (index_pred == index_gt).sum()
            if not vis:
                continue
            oppo_mesh = Fn.recon_error(oppo_x, mean, std, s, R, m, None, mesh=True)[2].cpu().numpy()
            recon_mesh, gt_np = res[3].cpu().numpy(), torch.as_tensor(gt_mesh).cpu().numpy()
            hit = (index_pred == index_gt).cpu().numpy()
            for i in range(len(names)):
                base = names[i].split("/")[-1].split(".")[0]
                d = ok_dir if hit[i] else bad_dir
                formats.save_obj(os.path.join(d, base + "_recon.obj"), recon_mesh[i], faces)
                formats.save_obj(os.path.join(d, base + "_gt.obj"), gt_np[i], faces)
                formats.save_obj(os.path.join(d, base + ".obj"), oppo_mesh[i], faces)
    r = meter.read()
    total = max(r["count"], 1)
    err = torch.cat(errors, 0).cpu().numpy() if errors else np.zeros((0, 0), dtype=np.float32)
    return r["loss"], r["kld"], r["rec_loss"], np.float64(r["accuracy"]), err, int(flipped) / total


def log_likelihood(model, loader, device, samples, sample_chunk=None, seed=0, log_sigma=None):
    """Held-out importance-weighted log-likelihood over a loader of the `evaluate` kind (`cheb_VAE.log_likelihood` per
    batch, each mesh under its own label, samples drawn from one device generator seeded with `seed`).  Nothing is read
    back before the end of the loop.  -> dict: per-mesh numpy fp64 arrays `log_px`, `elbo`, `ess`, their means
    `log_px_mean`, `elbo_mean`, `ess_mean`, and the meshes' file `names` in loader order.  Densities are those of the
    z-scored coordinates the model is trained on."""
    gen = torch.Generator(device=device)
    gen.manual_seed(int(seed))
    names_all, parts = [], []
    for data in loader:
        x, x_gt, y, names, _, _, _, _ = _split(data)
        x, x_gt = x.to(device, non_blocking=True), x_gt.to(device, non_blocking=True)
        y_hot = F.one_hot(y, num_classes=model.num_class).to(device, non_blocking=True)
        parts.append(torch.stack(model.log_likelihood(x, x_gt, y_hot, samples, sample_chunk, gen, log_sigma)))
        names_all += list(names)
    res = torch.cat(parts, 1).cpu().numpy() if parts else np.zeros((3, 0))
    out = {"names": names_all}
    for i, k in enumerate(("log_px", "elbo", "ess")):
        out[k] = res[i]
        out[k + "_mean"] = float(res[i].mean()) if res.shape[1] else float("nan")
    return out


def inference(net, output_path, mean, std, data_loader, faces, device, write_meshes=True):
    """inference.py:55-157 without its dataset construction: for every batch the predicted class of the (normalised)
    input, the reconstruction under that class and the sex-changed mesh under the opposite one; writes the
    `<name>_recon.obj` / `<name>_gt.obj` / `<name>.obj` triples into `output_path/sex_change` and the three reports
    `pred.json`, `error_list.json`, `inference.json` (formats.save_inference_reports).  The de-normalisation, the
    Procrustes back-transform and the per-mesh mean / max errors run on the device (`mvb_recon_error`); the meshes come
    back once per batch because they are written to disk.  -> the dict written to inference.json."""
    net.eval()
    mean, std = _norm(None, (mean, std), device)
    out_dir = os.path.join(output_path, "sex_change")
    os.makedirs(out_dir, exist_ok=True)
    names_all, sex_all, mean_all, max_all = [], [], [], []
    with torch.no_grad():
        for data in data_loader:
            x, x_gt, _, names, gt_mesh, R, m, s = _split(data)
            b = _num_graphs(x)
            x = x.to(device, non_blocking=True)
            x_gt = x_gt.to(device, non_blocking=True).reshape(b, -1, 3).float()          # inference.py:73
            pred = classifier_(net, x_gt)
            sex_hot = F.one_hot(pred, num_classes=2)
            _, _, out, z, _ = net(x, x_gt, sex_hot, m_type="test")
            res = Fn.recon_error(out, mean, std, s, R, m, gt_mesh, mesh=write_meshes)
            names_all += list(names)
            sex_all.append(pred)
            mean_all.append(res[0])
            max_all.append(res[1])
            if not write_meshes:
                continue
            oppo_x = net.sample(1 - sex_hot, z[2])
            oppo_mesh = Fn.recon_error(oppo_x, mean, std, s, R, m, None, mesh=True)[2].cpu().numpy()
            recon_mesh, gt_np = res[2].cpu().numpy(), torch.as_tensor(gt_mesh).cpu().numpy()
            for i in range(b):
                base = names[i].split("/")[-1].split(".")[0]
                formats.save_obj(os.path.join(out_dir, base + "_recon.obj"), recon_mesh[i], faces)
                formats.save_obj(os.path.join(out_dir, base + "_gt.obj"), gt_np[i], faces)
                formats.save_obj(os.path.join(out_dir, base + ".obj"), oppo_mesh[i], faces)
    sex = torch.cat(sex_all).cpu().numpy() if sex_all else np.zeros(0, dtype=np.int64)
    e_mean = torch.cat(mean_all).cpu().numpy() if mean_all else np.zeros(0)
    e_max = torch.cat(max_all).cpu().numpy() if max_all else np.zeros(0)
    formats.save_inference_reports(output_path, names_all, sex, e_mean, e_max)
    return {n.split("/").pop(): {"sex": int(sx), "reconstruction_error": {"mean": float(a), "max": float(c)}}
            for n, sx, a, c in zip(names_all, sex, e_mean, e_max)}


# ---- crecon.py: classifier on reconstruction residuals ---------------------------------------------------------
def estimate_diff(net, x, y, dtype, device=None):
    """crecon.py:162-201.  x [B,N,3] normalised meshes (or one [N,3] mesh), y [B] labels.  Encodes, classifies, decodes
    z_mean under the (true label when dtype == "train", else predicted) class and under the opposite one, and returns
    (cat(x - recon_opposite, x - recon_same) [B,N,6], number of correct class predictions as a device tensor)."""
    device = device if device is not None else next(net.parameters()).device
    ori = x
    if x.dim() == 2:
        x = x.reshape(1, -1, 3)
        ori = x
        y = torch.as_tensor(y).reshape(1)
    x, y = x.to(device), torch.as_tensor(y).to(device)
    ori = ori.to(device)
    with torch.no_grad():
        h = net.encoder(x)
        y_hat = net.classifier(h)
        index_pred = torch.argmax(y_hat, dim=1)
        correct = torch.sum(index_pred == y)
        sex_hot = F.one_hot(index_pred if dtype != "train" else y, num_classes=2)
        x_mean = net.z_mean(torch.cat([sex_hot, h], -1))
        recon = net.sample(sex_hot, x_mean)
        recon_oppo = net.sample(1 - sex_hot, x_mean)
        diff = torch.cat((ori - recon_oppo, ori - recon), dim=-1)
    return diff, correct


def train_classifier(model, dvae, train_loader, len_dataset, optimizer, device, criterion):
    """crecon.py:64-99 -> (summed batch losses / len_dataset, accuracy); totals stay on the device until the end"""
    model.train()
    dvae.eval()
    tot = torch.zeros(3, device=device, dtype=torch.float64)          # loss sum, correct, count
    for data in train_loader:
        _, x_gt, label, _, _, _, _, _ = _split(data)
        x_gt, label = x_gt.to(device, non_blocking=True).float(), label.to(device, non_blocking=True)
        diff, _ = estimate_diff(dvae, x_gt.reshape(label.shape[0], -1, 3), label, "train", device)
        optimizer.zero_grad()
        pred = model(diff)
        loss = criterion(pred, label)
        loss.backward()
        optimizer.step()
        predicted = torch.argmax(pred.detach(), dim=-1)               # argmax of the softmax (crecon.py:89)
        tot += torch.stack([loss.detach().double(), (predicted == label).sum().double(),
                            torch.tensor(float(label.shape[0]), device=device, dtype=torch.float64)])
    t = tot.cpu().numpy()
    return t[0] / len_dataset, t[1] / max(t[2], 1.0)


def evaluate_classifier(model, dvae, test_loader, len_dataset, device, criterion, err_file=False):
    """crecon.py:103-150 -> (loss, accuracy, {file name: predicted label} of the misclassified meshes if err_file)"""
    model.eval()
    dvae.eval()
    tot = torch.zeros(3, device=device, dtype=torch.float64)
    wrong = []
    with torch.no_grad():
        for data in test_loader:
            _, x_gt, label, names, _, _, _, _ = _split(data)
            x_gt, label = x_gt.to(device, non_blocking=True).float(), label.to(device, non_blocking=True)
            diff, _ = estimate_diff(dvae, x_gt.reshape(label.shape[0], -1, 3), label, "test", device)
            pred = model(diff)
            loss = criterion(pred, label)
            predicted = torch.argmax(pred, dim=-1)
            tot += torch.stack([loss.double(), (predicted == label).sum().double(),
                                torch.tensor(float(label.shape[0]), device=device, dtype=torch.float64)])
            if err_file:
                wrong.append((list(names), predicted, label))
    err = {}
    for names, predicted, label in wrong:                              # read back after the loop
        p, l = predicted.cpu().numpy().reshape(-1), label.cpu().numpy().reshape(-1)
        for i, name in enumerate(names):
            if p[i] != l[i]:
                err[name] = str(p[i])
    t = tot.cpu().numpy()
    return t[0] / len_dataset, t[1] / max(t[2], 1.0), err
