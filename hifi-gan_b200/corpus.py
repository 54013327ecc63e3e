"""Packed int16 training corpus: one file holding every training utterance, read through the page cache.

`train_loop` otherwise reads every training wav into host memory as fp32 and copies the concatenation to every GPU
(`SegmentSampler`), which does not fit LibriTTS-scale corpora.  A packed corpus stays on the host: `Corpus` maps it
read-only (`np.memmap`, so the ranks of a node share one page-cache copy) and `meldataset.CorpusSampler` sends each
batch's crops to the GPU.

Layout (little-endian; every section offset is a multiple of 4096):

    header   64 bytes   magic b"HGCORPUS", version, sampling_rate, num_mels (0: no mels), count,
                        index / names / pcm / mel section offsets
    index    count x _INDEX: sample offset, length, peak max|q|, mel frame offset, mel frames, name length
    names    utf-8 names, concatenated in index order
    pcm      int16 [sum length]                 the samples as the wav files hold them (channel 0)
    mel      fp32 [sum mel frames][num_mels]    fine-tuning mels, frame-major so that a crop is one contiguous run

Only 16-bit PCM wav files can be packed: the reference's `/ MAX_WAV_VALUE` convention assumes int16.  Float and
24-bit corpora keep using the in-memory `SegmentSampler`.

    python -m hifigan_b200.corpus --input_wavs_dir WAVS --input_training_file LIST --config CONFIG --output train.hgc
                                  [--input_mels_dir MELS]
"""
from __future__ import annotations

import argparse
import json
import os
import struct
from typing import Iterable, List, Optional, Tuple

import numpy as np

MAGIC = b"HGCORPUS"
VERSION = 1
PAGE = 4096
_HEADER = struct.Struct("<8sIIIIqqqqq")          # magic, version, sr, num_mels, reserved, count, 4 section offsets
_INDEX = np.dtype([("offset", "<i8"), ("length", "<i8"), ("mel_offset", "<i8"), ("mel_frames", "<i8"),
                   ("peak", "<i4"), ("name_len", "<i4")])


def _align(n: int) -> int:
    return (n + PAGE - 1) // PAGE * PAGE


def utterance_name(path: str) -> str:
    """The name a wav path is packed under: its file name without extension (what names its fine-tuning `.npy`)."""
    return os.path.splitext(os.path.split(path)[-1])[0]


def read_pcm16(path: str, sampling_rate: int) -> np.ndarray:
    """A 16-bit PCM wav file -> its int16 samples (channel 0).  Raises on a sampling-rate mismatch (the reference's
    message, meldataset.py:132-134) and on any other sample format."""
    from scipy.io.wavfile import read
    sr, data = read(path)
    if sr != sampling_rate:
        raise ValueError("{} SR doesn't match target {} SR".format(sr, sampling_rate))
    if data.dtype != np.int16:
        raise ValueError(f"{path}: {data.dtype} samples, not 16-bit PCM; only int16 wav files can be packed "
                         "(train float or 24-bit corpora from the wav files)")
    return data[:, 0] if data.ndim > 1 else data


def write(out_path: str, sampling_rate: int, names: List[str], utterances: Iterable[Tuple[np.ndarray, Optional[np.ndarray]]],
          ) -> None:
    """Write a corpus from `names` and one (int16 samples, fp32 mel [num_mels, F] or None) pair per name, consumed one
    at a time.  Either every utterance has a mel or none has."""
    n = len(names)
    blobs = [s.encode("utf-8") for s in names]
    index = np.zeros(n, _INDEX)
    index["name_len"] = [len(b) for b in blobs]
    index_off = _align(_HEADER.size)
    names_off = index_off + index.nbytes
    pcm_off = _align(names_off + sum(len(b) for b in blobs))
    num_mels, mel_tmp = 0, out_path + ".mels.tmp"
    pos = frames = count = 0
    with_mels = None
    with open(out_path, "wb") as f, open(mel_tmp, "w+b") as fm:
        try:
            f.seek(pcm_off)
            for i, (pcm, mel) in enumerate(utterances):
                if i >= n:
                    raise ValueError("more utterances than names")
                if with_mels is None:
                    with_mels = mel is not None
                elif with_mels != (mel is not None):
                    raise ValueError(f"{names[i]}: either every utterance has a fine-tuning mel or none has")
                pcm = np.ascontiguousarray(pcm, dtype=np.int16)
                index[i]["offset"], index[i]["length"] = pos, pcm.size
                index[i]["peak"] = int(np.abs(pcm.astype(np.int32)).max()) if pcm.size else 0
                f.write(pcm.tobytes())
                pos += pcm.size
                if mel is not None:
                    mel = np.asarray(mel, dtype=np.float32)
                    mel = mel.reshape(-1, mel.shape[-1])                      # [1, num_mels, F] or [num_mels, F]
                    if num_mels == 0:
                        num_mels = mel.shape[0]
                    elif mel.shape[0] != num_mels:
                        raise ValueError(f"{names[i]}: mel has {mel.shape[0]} bands, the first one {num_mels}")
                    index[i]["mel_offset"], index[i]["mel_frames"] = frames, mel.shape[1]
                    fm.write(np.ascontiguousarray(mel.T).tobytes())        # frame-major [F][num_mels]
                    frames += mel.shape[1]
                count += 1
            if count != n:
                raise ValueError(f"{count} utterances for {n} names")
            mel_off = _align(pcm_off + 2 * pos)
            if num_mels:
                f.seek(mel_off)
                fm.seek(0)
                while True:
                    chunk = fm.read(1 << 24)
                    if not chunk:
                        break
                    f.write(chunk)
            else:
                mel_off = 0
            f.truncate(max(f.tell(), pcm_off + 2 * pos))
            f.seek(0)
            f.write(_HEADER.pack(MAGIC, VERSION, sampling_rate, num_mels, 0, n, index_off, names_off, pcm_off, mel_off))
            f.seek(index_off)
            f.write(index.tobytes())
            f.write(b"".join(blobs))
        except BaseException:
            f.close()
            os.unlink(out_path)                # no half-written corpus is left behind
            raise
        finally:
            fm.close()
            os.unlink(mel_tmp)


def pack(wav_paths: List[str], out_path: str, sampling_rate: int, mels_dir: Optional[str] = None) -> None:
    """Pack 16-bit PCM wav files (and, with `mels_dir`, each one's fine-tuning mel `<mels_dir>/<name>.npy`) into one
    corpus file, reading one file at a time."""
    names = [utterance_name(p) for p in wav_paths]

    def items():
        for p, name in zip(wav_paths, names):
            mel = np.load(os.path.join(mels_dir, name + ".npy")) if mels_dir is not None else None
            yield read_pcm16(p, sampling_rate), mel
    write(out_path, sampling_rate, names, items())


class Corpus:
    """A packed corpus, mapped read-only.  `pcm` int16 [total samples] and `mels` fp32 [total frames][num_mels] (None
    without fine-tuning mels) are views of the mapping; the per-utterance arrays are int64 numpy arrays."""

    def __init__(self, path: str):
        self.path = path
        self._map = np.memmap(path, dtype=np.uint8, mode="r")
        if self._map.size < _HEADER.size:
            raise ValueError(f"{path}: not a packed corpus (too short)")
        magic, version, sr, num_mels, _, n, index_off, names_off, pcm_off, mel_off = _HEADER.unpack(
            self._map[:_HEADER.size].tobytes())
        if magic != MAGIC or version != VERSION:
            raise ValueError(f"{path}: not a packed corpus (version {VERSION})")
        self.sampling_rate, self.num_mels = sr, num_mels
        index = np.frombuffer(self._map, _INDEX, count=n, offset=index_off)
        self.offsets = index["offset"].astype(np.int64)
        self.lengths = index["length"].astype(np.int64)
        self.peaks = index["peak"].astype(np.int64)
        self.mel_offsets = index["mel_offset"].astype(np.int64)
        self.mel_frames = index["mel_frames"].astype(np.int64)
        blob = self._map[names_off:names_off + int(index["name_len"].sum())].tobytes()
        ends = np.cumsum(index["name_len"])
        self.names = [blob[e - k:e].decode("utf-8") for e, k in zip(ends.tolist(), index["name_len"].tolist())]
        total = int(self.lengths.sum())
        self.pcm = self._map[pcm_off:pcm_off + 2 * total].view(np.int16)
        self.mels = None
        if num_mels:
            nf = int(self.mel_frames.sum())
            self.mels = self._map[mel_off:mel_off + 4 * nf * num_mels].view(np.float32).reshape(nf, num_mels)

    def __len__(self) -> int:
        return len(self.names)

    def samples(self, i: int) -> np.ndarray:
        o = int(self.offsets[i])
        return self.pcm[o:o + int(self.lengths[i])]

    def mel(self, i: int) -> np.ndarray:
        """Fine-tuning mel of utterance i, frame-major [F][num_mels]."""
        o = int(self.mel_offsets[i])
        return self.mels[o:o + int(self.mel_frames[i])]


def main(argv=None) -> None:
    from .meldataset import read_filelist
    parser = argparse.ArgumentParser(description="Pack the 16-bit PCM training wav files of a file list into one corpus")
    parser.add_argument('--input_wavs_dir', default='LJSpeech-1.1/wavs')
    parser.add_argument('--input_training_file', default='LJSpeech-1.1/training.txt')
    parser.add_argument('--input_mels_dir', default=None, help="fine-tuning mels <name>.npy to pack with the audio")
    parser.add_argument('--config', required=True)
    parser.add_argument('--output', required=True)
    a = parser.parse_args(argv)
    with open(a.config) as f:
        h = json.load(f)
    paths = read_filelist(a.input_training_file, a.input_wavs_dir)
    pack(paths, a.output, h["sampling_rate"], a.input_mels_dir)
    c = Corpus(a.output)
    print(f"{a.output}: {len(c)} utterances, {c.pcm.size} samples at {c.sampling_rate} Hz"
          + (f", {c.mels.shape[0]} mel frames" if c.mels is not None else ""))


if __name__ == "__main__":
    main()
