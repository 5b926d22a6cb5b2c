"""Scenes at the tracker's capacity corners, shared by the CPU (host emulation) and GPU tests: a crowd of about a
thousand objects (most shrunk to fit the scene's box, a few large and slow so that their tracks gate many
detections), and 128 labels whose name order differs from their index order, counted on 32 lines with exact vote
ties and the motorbike/bicycle rule at high label indices."""
import numpy as np
import torch

from deepdish_b200.scene import Scene
from oracle import countline as oc

# 126 names in an order unrelated to their index ((37 k) mod 128 is a permutation), then motorbike and bicycle at the
# two highest indices (their names sort between the others)
LABELS128 = ["c%03d" % ((37 * k) % 128) for k in range(126)] + ["motorbike", "bicycle"]
MOTORBIKE, BICYCLE = 126, 127
# 32 count lines: 16 vertical and 16 horizontal, so that most moving tracks cross some line every few ticks
LINES32 = np.array([(20.0 + 38.0 * k, 0.0, 20.0 + 38.0 * k, 480.0) for k in range(16)]
                   + [(0.0, 12.0 + 28.0 * k, 640.0, 12.0 + 28.0 * k) for k in range(16)], np.float64)


def crowd(n_objects, dmax, seed, big=60, miss_prob=0.04):
    """A Scene of n_objects in the usual 600 x 400 box: boxes shrunk to 0.3 of their size and speed, except the first
    `big` objects, four times their size and a fifth of their speed (tracks that pass many detections' gates)."""
    sc = Scene(1, n_objects, dmax, n_labels=3, seed=seed, miss_prob=miss_prob)
    size = torch.full((1, n_objects, 1), 0.3)
    size[:, :big] = 4.0
    vel = torch.full((1, n_objects, 1), 0.3)
    vel[:, :big] = 0.2
    sc.size, sc.vel = sc.size * size, sc.vel * vel
    return sc


class LabelScene:
    """Scene over LABELS128 whose batches carry one confidence for every detection (so two labels seen equally often
    by a track tie exactly in its vote, and the name order decides), and in which the objects of labels 0..31 are
    reported as motorbike or bicycle (the rule of track.py:175-183)."""

    def __init__(self, n_streams, n_objects, dmax, seed):
        self.sc = Scene(n_streams, n_objects, dmax, n_labels=128, seed=seed, label_noise=0.3)
        self.gen = torch.Generator().manual_seed(seed)

    def step(self):
        b = self.sc.step()
        b.conf = torch.full_like(b.conf, 0.75)
        two = b.label < 32
        bike = torch.rand(b.label.shape, generator=self.gen) < 0.35
        b.label = torch.where(two, torch.where(bike, BICYCLE, MOTORBIKE), b.label).to(torch.int32)
        return b


def line_counters(n_streams, labels=LABELS128, lines=LINES32):
    """One oracle LineCounter per stream and line."""
    return [[oc.LineCounter(np.asarray(l, float).reshape(2, 2), labels) for l in lines] for _ in range(n_streams)]


def line_counts(counters, labels=LABELS128):
    """[S, L, C, 4] counters of line_counters."""
    return np.array([[c.counts(labels) for c in cs] for cs in counters], np.int64)


def vote_corners(trackers):
    """(tracks whose vote is an exact tie between their two leading labels, tracks whose vote leads with motorbike
    over bicycle) among the live tracks of the oracle trackers."""
    ties = rule = 0
    for trk in trackers:
        for t in trk.tracks:
            if len(t.dist) < 2:
                continue
            cnt = np.array([len(s) for s in t.dist.values()])
            alphas = np.array([np.average(s) for s in t.dist.values()])
            v = (alphas + cnt) / (cnt.sum() + alphas.sum())
            ranked = sorted(zip(v, t.dist.keys()), reverse=True)
            ties += ranked[0][0] == ranked[1][0]
            rule += ranked[0][1] == "motorbike" and ranked[1][1] == "bicycle"
    return ties, rule
