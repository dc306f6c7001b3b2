"""Host-side mirror of the reference worker script `ssgd_monitor.py` (shifu-tensorflow-on-yarn/src/main/resources/),
the plug-in the stock YARN executor launches through `shifu.application.python-script-path`
(TensorflowTaskExecutor.java:273-275, 300-317).  Same seam, same names, same contract:

  env in    JOB_NAME, TASK_ID, WORKER_CNT, CLUSTER_SPEC, TRAINING_DATA_PATH, TOTAL_TRAINING_DATA_NUMBER,
            SELECTED_COLUMN_NUMS, WEIGHT_COLUMN_NUM, TARGET_COLUMN_NUM, TMP_MODEL_PATH, FINAL_MODEL_PATH,
            SOCKET_SERVER_PORT                                   (ssgd_monitor.py:36-50)
  files in  ./ModelConfig.json  (train.params.NumHiddenLayers / NumHiddenNodes / ActivationFunc / LearningRate,
            train.numTrainEpochs, train.validSetRate; ssgd_monitor.py:92-95,133,178-183)
  out       one line per epoch on 127.0.0.1:$SOCKET_SERVER_PORT
            "worker_index:{},time:{},current_epoch:{},training_loss:{},valid_loss:{}\n"   (ssgd_monitor.py:288-293,
            parsed by SocketServer.java:71-89); SavedModel + GenericModelConfig.json at FINAL_MODEL_PATH (chief);
            exit code 0

What changed underneath: the TF graph / Session / parameter servers are gone.  All arithmetic is the CUDA library
behind the C-ABI (`_capi.Trainer`); workers are data-parallel ranks that exchange gradients over NCCL, `JOB_NAME=ps`
processes simply idle (the stock AM insists on >= 1 PS, SURVEY.md 8b).  The reference's `time.sleep(40)` grace
periods and the 5 s sleep per epoch are not reproduced.

Optional ModelConfig train.params the reference does not have (defaults = reference behaviour):
  Optimizer  "adadelta" (default) | "adam" | "sgd" | "momentum"
  Loss       "squared" (default: MSE on the sigmoid output, ssgd_monitor.py:129) | "log" (sigmoid cross-entropy)
  Precision  "bf16" (default) | "fp32" (CUDA-core parity mode) | "fp32_tc" (fp32-class accuracy on the tensor cores:
             three bf16 parts per value) | "bf16x2" (two parts)
  MiniBatchs mini-batch rows (default BATCH_SIZE = 100, ssgd_monitor.py:33)
  Schedule   "sync_replicas" (default; "epoch" is accepted as an alias): the reference's SyncReplicasOptimizer schedule
             (ssgd_monitor.py:136-141,218,259-260) - every run pushes its mini-batch gradient, a push tagged with a stale
             local step is dropped, after R = replicas_to_aggregate accepted pushes their MEAN is applied as ONE update
             (class SyncReplicasSchedule below restates the token / accumulator bookkeeping on the host)
             | "batch" (one update per mini-batch, the north-star wording)

File paths (TRAINING_DATA_PATH, TMP_MODEL_PATH, FINAL_MODEL_PATH) may carry a scheme.  The stock AM hands out fully
qualified HDFS URIs (TrainingDataSet.java:74) which the reference reads through tf.gfile; here `hdfs://`, `viewfs://`,
`webhdfs://`, `s3a://` ... go through the `hdfs dfs` command line of the container (class _Fs), `file://` and plain
paths are local, and the checkpoint / SavedModel are staged locally and uploaded.  A scheme path without a usable
`hdfs` binary fails fast with a clear message instead of a FileNotFoundError deep inside the loader.
"""
from __future__ import annotations

import gzip
import io
import json
import logging
import os
import random
import shutil
import socket
import struct
import subprocess
import sys
import tempfile
import time
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _capi as capi

HIDDEN_NODES_COUNT = 20
VALID_TRAINING_DATA_RATIO = 0.1
BUILD_MODEL_BY_CONF_ENABLE = True
REPLICAS_TO_AGGREGATE_RATIO = 1
DELIMITER = '|'
BATCH_SIZE = 100

_OPT = {"adadelta": capi.OPT_ADADELTA, "adam": capi.OPT_ADAM, "sgd": capi.OPT_SGD, "momentum": capi.OPT_MOMENTUM}
_LOSS = {"squared": capi.LOSS_MSE, "log": capi.LOSS_SIGMOID_CE}


def get_activation_fun(name: Optional[str]) -> int:
    """name -> activation id; None / unknown -> leaky_relu (ssgd_monitor.py:74-88)."""
    if name is None:
        return capi.ACT_LEAKYRELU
    name = name.lower()
    if 'sigmoid' == name:
        return capi.ACT_SIGMOID
    elif 'tanh' == name:
        return capi.ACT_TANH
    elif 'relu' == name:
        return capi.ACT_RELU
    elif 'leakyrelu' == name:
        return capi.ACT_LEAKYRELU
    else:
        return capi.ACT_LEAKYRELU


def generate_from_modelconf(model_conf: dict):
    """-> (hidden widths, activation ids) (ssgd_monitor.py:91-107)."""
    train_params = model_conf['train']['params']
    num_hidden_layer = int(train_params['NumHiddenLayers'])
    num_hidden_nodes = [int(s) for s in train_params['NumHiddenNodes']]
    activation_func = [get_activation_fun(s) for s in train_params['ActivationFunc']]
    return num_hidden_nodes[:num_hidden_layer], activation_func[:num_hidden_layer]


def model(feature_count: int, model_conf: Optional[dict], max_batch: int) -> capi.NetDesc:
    """The network + loss + optimizer of `model()` (ssgd_monitor.py:110-144) as a C-ABI net descriptor."""
    if BUILD_MODEL_BY_CONF_ENABLE and model_conf is not None:
        hidden, acts = generate_from_modelconf(model_conf)
        params = model_conf['train']['params']
        learning_rate = float(params['LearningRate'])
    else:
        hidden, acts, params = [HIDDEN_NODES_COUNT], [capi.ACT_TANH], {}
        learning_rate = 0.003
    opt = _OPT[str(params.get('Optimizer', 'adadelta')).lower()]
    loss = _LOSS[str(params.get('Loss', 'squared')).lower()]
    prec = {'fp32': capi.PREC_FP32, 'fp32_tc': capi.PREC_FP32_TC, 'bf16x2': capi.PREC_BF16X2}.get(
        str(params.get('Precision', 'bf16')).lower(), capi.PREC_BF16)
    return capi.make_desc(feature_count, hidden, acts, loss=loss, optimizer=opt, learning_rate=learning_rate,
                          max_batch=max_batch, precision=prec)


class _Fs:
    """tf.gfile stand-in: local paths directly, scheme paths through `hdfs dfs` (present in every YARN container)."""
    CLI = os.environ.get("SB_HDFS_CLI", "hdfs")

    @staticmethod
    def is_remote(path: str) -> bool:
        return "://" in path and not path.startswith("file://")

    @staticmethod
    def local(path: str) -> str:
        return path[len("file://"):] if path.startswith("file://") else path

    @classmethod
    def _run(cls, args: List[str], what: str, capture: bool = False):
        try:
            r = subprocess.run([cls.CLI, "dfs"] + args, stdout=subprocess.PIPE if capture else subprocess.DEVNULL,
                               stderr=subprocess.PIPE)
        except FileNotFoundError:
            raise RuntimeError("%s needs the `%s` command on PATH (set SB_HDFS_CLI), or use a local / NFS path" % (what, cls.CLI))
        if r.returncode != 0:
            raise IOError("%s failed (%s dfs %s): %s" % (what, cls.CLI, " ".join(args), r.stderr.decode("utf8", "replace").strip()))
        return r.stdout

    @classmethod
    def read_bytes(cls, path: str) -> bytes:
        if cls.is_remote(path):
            return cls._run(["-cat", path], "reading " + path, capture=True)
        with open(cls.local(path), 'rb') as f:
            return f.read()

    @classmethod
    def exists(cls, path: str) -> bool:
        if not cls.is_remote(path):
            return os.path.exists(cls.local(path))
        try:
            cls._run(["-test", "-e", path], "probing " + path)
            return True
        except IOError:
            return False

    @classmethod
    def fetch(cls, path: str, local_dst: str) -> None:
        cls._run(["-get", "-f", path, local_dst], "downloading " + path)

    @classmethod
    def upload(cls, local_src: str, path: str, replace_dir: bool = False) -> None:
        if replace_dir:
            try:
                cls._run(["-rm", "-r", "-f", path], "replacing " + path)
            except IOError:
                pass
        parent = path.rstrip("/").rsplit("/", 1)[0]
        cls._run(["-mkdir", "-p", parent], "creating " + parent)
        cls._run(["-put", "-f", local_src, path], "uploading " + path)


def load_data(data_file: str, feature_column_nums: Optional[List[int]], target_column_num: int,
              sample_weight_column_num: int, valid_ratio: float, rng=random) -> Dict[str, object]:
    """Same semantics as the reference loader (ssgd_monitor.py:348-454): comma-separated list of gzip files, '|'
    delimited lines, selected columns -> float (an unparsable cell is logged and skipped, :409-411), weight < 0 -> 1.0,
    no weight column -> 1.0, Bernoulli(valid_ratio) split by `random.random() >= ratio -> train` (:396)."""
    out = {k: [] for k in ("train_data", "train_target", "valid_data", "valid_target",
                           "train_data_sample_weight", "valid_data_sample_weight")}
    line_count = 0
    for current_file in data_file.split(","):
        logging.info("Now loading " + current_file)
        gf = gzip.GzipFile(fileobj=io.BytesIO(_Fs.read_bytes(current_file)))
        for raw in gf:
            line = raw.decode('utf-8')
            if len(line) == 0:
                break
            line_count += 1
            columns = line.split(DELIMITER)
            if feature_column_nums is None:
                feature_column_nums = [c for c in range(len(columns)) if c != target_column_num and
                                       not (sample_weight_column_num >= 0 and c == sample_weight_column_num)]
            pre = "train" if rng.random() >= valid_ratio else "valid"
            out[pre + "_target"].append([float(columns[target_column_num])])
            row = []
            for c in feature_column_nums:
                try:
                    row.append(float(columns[c].strip('\n')))
                except Exception:
                    logging.info("Could not convert " + str(columns[c].strip('\n')) + " to float")
                    logging.info("feature_column_num: " + str(c))
            out[pre + "_data"].append(row)
            if 0 <= sample_weight_column_num < len(columns):
                weight = float(columns[sample_weight_column_num].strip('\n'))
                if weight < 0.0:
                    logging.info("Warning: weight is below 0. example:" + line)
                    weight = 1.0
                out[pre + "_data_sample_weight"].append([weight])
            else:
                out[pre + "_data_sample_weight"].append([1.0])
    logging.info("Total data count: " + str(line_count) + ".")
    out["feature_count"] = len(feature_column_nums) if feature_column_nums is not None else 0
    return out


def load_data_gpu(data_file: str, feature_column_nums: Optional[List[int]], target_column_num: int,
                  sample_weight_column_num: int, valid_ratio: float, rng=random, device: int = 0) -> Dict[str, object]:
    """load_data with the per-cell float() loop moved to the GPU (sb_text_parse): the host only gunzips and draws the
    train/valid coin per line (same `rng.random() >= ratio -> train` stream, ssgd_monitor.py:396); cells the exact
    fast path declines come back as a list and are resolved with float() here, exactly like the reference would.
    Returns capi.DeviceArray objects under the same keys as load_data: the parsed set never visits the host (the trainer's
    load_dataset / eval_loss take device pointers)."""
    chunks = []
    for current_file in data_file.split(","):
        data = gzip.GzipFile(fileobj=io.BytesIO(_Fs.read_bytes(current_file))).read()
        if data and not data.endswith(b"\n"):
            data += b"\n"
        chunks.append(data)
    text = b"".join(chunks)
    first = text[:text.index(b"\n")].decode('utf-8').split(DELIMITER)
    if feature_column_nums is None:
        feature_column_nums = [c for c in range(len(first)) if c != target_column_num and
                               not (sample_weight_column_num >= 0 and c == sample_weight_column_num)]
    n_map = max([target_column_num, sample_weight_column_num] + list(feature_column_nums)) + 1
    col_map = [capi.COL_SKIP] * n_map
    for j, c in enumerate(feature_column_nums):
        col_map[c] = j
    col_map[target_column_num] = capi.COL_TARGET
    if sample_weight_column_num >= 0:
        col_map[sample_weight_column_num] = capi.COL_WEIGHT
    n_feat = len(feature_column_nums)
    X, y, w, flags, text, _kernel_ms = capi.text_parse_device(text, col_map, n_feat, DELIMITER, device=device)
    for row, slot, off, ln in flags:
        if slot == -100:
            raise ValueError("line %d does not have the selected columns" % row)
        cell = text[off:off + ln].decode('utf-8')
        v = float(cell.strip('\n'))        # ValueError here = the cell the reference would log and skip
        if slot >= 0:
            X.patch(row * n_feat + slot, v)
        elif slot == capi.COL_TARGET:
            y.patch(row, v)
        else:
            w.patch(row, 1.0 if v < 0.0 else v)
    # the Bernoulli coins come from the caller's RNG (one draw per line, in line order, like the reference); only the row
    # indices of the two sides travel to the device, the parsed set itself stays there
    coins = np.fromiter((rng.random() >= valid_ratio for _ in range(len(y))), dtype=bool, count=len(y))
    tr_rows, va_rows = np.flatnonzero(coins), np.flatnonzero(~coins)
    out = {"feature_count": n_feat}
    for pre, rows in (("train", tr_rows), ("valid", va_rows)):
        out[pre + "_data"] = X.take_rows(rows)
        out[pre + "_target"] = y.take_rows(rows)
        out[pre + "_data_sample_weight"] = w.take_rows(rows)
    for a in (X, y, w):
        a.free()
    return out


def simple_save(trainer: capi.Trainer, export_dir: str) -> None:
    """SavedModel (tag serve, signature serving_default shifu_input_0 -> shifu_output_0) + GenericModelConfig.json
    (ssgd_monitor.py:457-490); an existing export_dir is replaced like tf.gfile.DeleteRecursively does."""
    if _Fs.is_remote(export_dir):
        stage = tempfile.mkdtemp(prefix="sb_export_")
        try:
            local = os.path.join(stage, "model")
            trainer.export_savedmodel(local)
            _Fs.upload(local, export_dir, replace_dir=True)
        finally:
            shutil.rmtree(stage, ignore_errors=True)
        return
    export_dir = _Fs.local(export_dir)
    if os.path.exists(export_dir):
        shutil.rmtree(export_dir)
    trainer.export_savedmodel(export_dir)


class Rendezvous:
    """The host-side channel that replaces tf.train.Server / ClusterSpec (ssgd_monitor.py:152-166): worker 0 listens ONCE
    on its own CLUSTER_SPEC address (the port the executor reserved for TF, TensorflowTaskExecutor.java:93-111), every
    other worker connects once, and the connections stay open for every later round (NCCL id, IPC handles, ok flags).
    Rounds are tagged, every socket operation has a deadline, so a worker that died is an error here instead of a hang."""

    def __init__(self, cluster_spec: dict, task_index: int, n_workers: int, timeout: float = 1200.0):
        # 1200 s: the AM gives stragglers 20 min before it fails the job (Constants.java:92-94)
        self.rank, self.n, self.timeout, self.round = task_index, n_workers, timeout, 0
        self.conns: Dict[int, socket.socket] = {}
        self.hub: Optional[socket.socket] = None
        if n_workers <= 1:
            return
        host, port = cluster_spec['worker'][0].rsplit(':', 1)
        port = int(port)
        deadline = time.time() + timeout
        if task_index == 0:
            srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
            srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
            srv.bind(('', port))
            srv.listen(n_workers)
            try:
                while len(self.conns) < n_workers - 1:
                    srv.settimeout(max(0.1, deadline - time.time()))
                    try:
                        conn, _addr = srv.accept()
                    except socket.timeout:
                        missing = sorted(set(range(1, n_workers)) - set(self.conns))
                        raise RuntimeError("rendezvous: workers %s did not connect within %.0f s" % (missing, timeout))
                    conn.settimeout(timeout)
                    (r,) = struct.unpack("<i", _recv_exact(conn, 4))
                    self.conns[r] = conn
            finally:
                srv.close()
        else:
            while True:
                try:
                    c = socket.create_connection((host, port), timeout=10)
                    break
                except OSError:
                    if time.time() > deadline:
                        raise RuntimeError("rendezvous: worker 0 at %s:%d unreachable for %.0f s" % (host, port, timeout))
                    time.sleep(0.2)
            c.settimeout(timeout)
            c.sendall(struct.pack("<i", task_index))
            self.hub = c

    def allgather(self, payload: bytes) -> List[bytes]:
        """every worker contributes one byte string, every worker gets all of them in rank order"""
        if self.n <= 1:
            return [payload]
        self.round += 1
        if self.rank == 0:
            parts: Dict[int, bytes] = {0: payload}
            for r, conn in self.conns.items():
                rnd, size = struct.unpack("<ii", _recv_exact(conn, 8))
                if rnd != self.round:
                    raise RuntimeError("rendezvous: worker %d is in round %d, worker 0 in round %d" % (r, rnd, self.round))
                parts[r] = _recv_exact(conn, size)
            blob = b"".join(struct.pack("<i", len(parts[r])) + parts[r] for r in range(self.n))
            for conn in self.conns.values():
                conn.sendall(blob)
            return [parts[r] for r in range(self.n)]
        self.hub.sendall(struct.pack("<ii", self.round, len(payload)) + payload)
        out = []
        for _ in range(self.n):
            (size,) = struct.unpack("<i", _recv_exact(self.hub, 4))
            out.append(_recv_exact(self.hub, size))
        return out

    def bcast(self, payload: Optional[bytes]) -> bytes:
        """worker 0's payload on every worker"""
        return self.allgather(payload if self.rank == 0 and payload is not None else b"")[0]

    def close(self):
        for c in list(self.conns.values()) + ([self.hub] if self.hub is not None else []):
            try:
                c.close()
            except OSError:
                pass
        self.conns, self.hub = {}, None


def _recv_exact(c: socket.socket, n: int) -> bytes:
    buf = b""
    while len(buf) < n:
        chunk = c.recv(n - len(buf))
        if not chunk:
            raise RuntimeError("rendezvous: connection closed")
        buf += chunk
    return buf


def exchange_nccl_id(rdv: Rendezvous) -> Optional[bytes]:
    """worker 0 creates the 128-byte NCCL unique id, every worker gets it"""
    if rdv.n <= 1:
        return None
    return rdv.bcast(capi.nccl_unique_id() if rdv.rank == 0 else None)


def enable_peer_exchange(trainer, rdv: Rendezvous) -> bool:
    """When every rank runs on this host (launcher.py: one rank per GPU of the node), switch the gradient exchange from
    NCCL to the peer-memory kernels: all-gather (hostname, CUDA-IPC handle), map the peers (sb_trainer_set_peer_handles),
    then all-gather an ok flag - the switch only happens if EVERY rank mapped every peer (cudaIpcOpenMemHandle fails
    without P2P / NVLink, across IPC namespaces, or on distinct hosts that share a hostname); otherwise every rank
    drops its mappings again and NCCL stays.  Returns whether the peer exchange is on."""
    n = rdv.n
    if n <= 1 or n > 16:
        return False
    me = socket.gethostname().encode("utf8")
    got = rdv.allgather(struct.pack("<H", len(me)) + me + trainer.ipc_handle())
    hosts, handles = [], []
    for b in got:
        (k,) = struct.unpack("<H", b[:2])
        hosts.append(b[2:2 + k]); handles.append(b[2 + k:])
    if len(set(hosts)) != 1:
        return False
    ok, why = True, ""
    try:
        trainer.set_peer_handles(handles)
    except Exception as e:          # noqa: BLE001 - any failure here means "keep NCCL", never "crash the job"
        ok, why = False, str(e)
    flags = rdv.allgather(b"\x01" if ok else b"\x00" + why.encode("utf8", "replace")[:200])
    if all(f[:1] == b"\x01" for f in flags):
        return True
    bad = ["worker %d: %s" % (r, f[1:].decode("utf8", "replace")) for r, f in enumerate(flags) if f[:1] != b"\x01"]
    logging.warning("peer-memory exchange unavailable, staying on NCCL (%s)" % "; ".join(bad))
    if ok and hasattr(trainer, "clear_peer_handles"):
        trainer.clear_peer_handles()
    return False


class SyncReplicasSchedule:
    """Host bookkeeping of tf.train.SyncReplicasOptimizer + ConditionalAccumulator as the reference drives them
    (ssgd_monitor.py:136-142 builds it with replicas_to_aggregate = R, :218/:259-260 seed R tokens valued 0, every
    sess.run(train_step) :276 pushes then dequeues).  TF-library semantics, restated (not in the reference tree): a push
    carries the worker's local_step and is DROPPED when that is older than the accumulator's step; after R accepted
    pushes their mean is applied once, global_step += 1 and R tokens valued global_step are enqueued; every run ends by
    dequeuing one token, which becomes the worker's local_step.

    All workers step in lock-step here (one synchronous exchange per round), so "arrival order" is rank order within a
    round; with one worker this is exactly oracle/shifu_oracle.py:SyncReplicasTrainer.  Every rank runs the same
    deterministic bookkeeping for ALL ranks, so no extra communication is needed to agree on who was accepted.

    A worker whose dequeue finds the token queue empty BLOCKS inside its sess.run until the next update enqueues tokens
    (served first come, first served); while blocked it issues no further runs.

    round() -> (ran, accepted, apply, pushes)
        ran[r]       rank r executes a run in this round (False: it is still blocked in its previous run's dequeue)
        accepted[r]  rank r's gradient of this round counts (else the run only reports its loss)
        apply        the accumulator filled in this round: apply the mean of `pushes` (= R) accepted gradients now"""

    def __init__(self, R: int, n_workers: int = 1):
        self.R, self.n = max(1, int(R)), max(1, int(n_workers))
        self.global_step = 0
        self.local_step = [0] * self.n
        self.tokens: List[int] = [0] * self.R
        self.acc_n = 0
        self.waiting: List[int] = []          # ranks blocked in the token dequeue, in arrival order

    def _serve(self):
        while self.waiting and self.tokens:
            self.local_step[self.waiting.pop(0)] = self.tokens.pop(0)

    def round(self):
        blocked = set(self.waiting)
        ran = [r not in blocked for r in range(self.n)]
        if not any(ran):
            raise RuntimeError("every worker is blocked on the sync token queue: the reference would hang here "
                               "(replicas_to_aggregate=%d, %d workers)" % (self.R, self.n))
        accepted, apply_now, pushes = [False] * self.n, False, 0
        for r in range(self.n):
            if not ran[r]:
                continue
            if self.local_step[r] >= self.global_step:       # a push tagged with an older step is dropped
                accepted[r] = True
                self.acc_n += 1
            if self.acc_n >= self.R:                          # take_grad(R): at most once per round, later pushes are stale
                apply_now, pushes = True, self.acc_n
                self.acc_n = 0
                self.global_step += 1
                self.tokens.extend([self.global_step] * self.R)
                self._serve()
            self.waiting.append(r)                            # dequeue one token (or block until there is one)
            self._serve()
        return ran, accepted, apply_now, pushes


def row_shard(spec: str, *arrays):
    """spec "g/G": rows g::G of every array, truncated to len // G rows (identical on all G ranks)"""
    g, G = (int(v) for v in spec.split("/"))
    if not (0 <= g < G):
        raise ValueError("SB_ROW_SHARD must be g/G with 0 <= g < G, got %r" % spec)
    n = len(arrays[0]) // G
    return tuple(np.ascontiguousarray(a[g::G][:n]) for a in arrays)


def equal_size_runs(bounds):
    """bounds = batch start offsets + [n_rows] (np.array_split: sizes differ by at most one row) ->
    [(first batch index, number of consecutive batches, rows per batch)]"""
    runs, i, nb = [], 0, len(bounds) - 1
    while i < nb:
        rows = int(bounds[i + 1] - bounds[i])
        j = i
        while j < nb and int(bounds[j + 1] - bounds[j]) == rows:
            j += 1
        runs.append((i, j - i, rows))
        i = j
    return runs


def main(_=None, env=None, rng=random) -> int:
    env = os.environ if env is None else env
    logging.basicConfig(level=logging.INFO, format='%(asctime)s %(name)-12s %(levelname)-8s %(message)s',
                        datefmt='%y-%m-%d %H:%M:%S')
    # read from env (ssgd_monitor.py:36-50) - a missing key raises KeyError exactly like the reference
    cluster_spec = json.loads(env["CLUSTER_SPEC"])
    n_workers = int(env["WORKER_CNT"])
    job_name = env["JOB_NAME"]
    task_index = int(env["TASK_ID"])
    socket_server_port = int(env["SOCKET_SERVER_PORT"])
    total_training_data_number = int(env["TOTAL_TRAINING_DATA_NUMBER"])
    # Column lists: SELECTED_COLUMN_NUMS, or - when the job configuration leaves it blank - the numeric / categorical pair the
    # executor exports instead (TensorflowTaskExecutor.java:213-223).  The reference script only ever reads the first and dies
    # with a KeyError on the second form; here the pair selects the wide+deep model (BASELINE config 4, oracle/wide_deep.py):
    # numeric columns -> dense block, categorical columns -> integer codes 0 .. V_c-1 (anything else = missing) whose one-hot
    # expansion is evaluated as an embedding gather.
    numeric_cols = [int(v) for v in str(env.get("SELECTED_NUMERIC_COLUMN_NUMS", "")).split() if int(v) >= 0]
    category_cols = [int(v) for v in str(env.get("SELECTED_CATEGORY_COLUMN_NUMS", "")).split() if int(v) >= 0]
    sel = str(env.get("SELECTED_COLUMN_NUMS", "")).strip()
    wide_deep = (sel in ("", "-1")) and bool(numeric_cols) and bool(category_cols)
    if wide_deep:
        feature_column_nums = numeric_cols + category_cols
    else:
        feature_column_nums = [int(s) for s in str(env["SELECTED_COLUMN_NUMS"]).split(' ')]
    feature_count = len(feature_column_nums)
    sample_weight_column_num = int(env["WEIGHT_COLUMN_NUM"])
    target_column_num = int(env["TARGET_COLUMN_NUM"])
    tmp_model_path = env["TMP_MODEL_PATH"]
    final_model_path = env["FINAL_MODEL_PATH"]
    logging.info("job_name:%s, task_index:%d" % (job_name, task_index))

    if job_name == 'ps':
        # server.join() (ssgd_monitor.py:157-161): there is no parameter server any more; idle until YARN reaps us
        while True:
            time.sleep(3600)

    socket_client = None
    try:
        socket_client = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
        socket_client.connect(("127.0.0.1", socket_server_port))
    except OSError:
        if env.get("SB_REQUIRE_SOCKET", "1") != "0":
            raise
        socket_client = None
    is_chief = (task_index == 0)
    training_data_path = env["TRAINING_DATA_PATH"]

    with open('./ModelConfig.json') as f:
        model_conf = json.load(f)
    epochs = int(model_conf['train']['numTrainEpochs'])
    valid_ratio = model_conf['train']['validSetRate']
    params = model_conf['train']['params']
    batch_size = int(params.get('MiniBatchs', BATCH_SIZE))
    schedule = str(params.get('Schedule', 'sync_replicas')).lower()
    if schedule not in ('sync_replicas', 'epoch', 'batch'):
        raise ValueError("train.params.Schedule must be sync_replicas (alias epoch) or batch, got %r" % schedule)
    per_batch_update = schedule == 'batch'

    device = int(env.get("SB_DEVICE", env.get("LOCAL_RANK", "0")))
    if env.get("SB_HOST_LOADER", "0") == "1":
        context = load_data(training_data_path, feature_column_nums, target_column_num, sample_weight_column_num,
                            valid_ratio, rng=rng)
    else:
        context = load_data_gpu(training_data_path, feature_column_nums, target_column_num, sample_weight_column_num,
                                valid_ratio, rng=rng, device=device)
    on_device = isinstance(context["train_data"], capi.DeviceArray)
    if on_device:
        train_x, train_y, train_w = context["train_data"], context["train_target"], context["train_data_sample_weight"]
        valid_x, valid_y, valid_w = context["valid_data"], context["valid_target"], context["valid_data_sample_weight"]
        if len(train_x.shape) != 2 or train_x.shape[1] != feature_count:
            raise ValueError("training rows do not all have %d parsable features" % feature_count)
        if env.get("SB_ROW_SHARD"):
            g, G = (int(v) for v in env["SB_ROW_SHARD"].split("/"))
            if not (0 <= g < G):
                raise ValueError("SB_ROW_SHARD must be g/G with 0 <= g < G, got %r" % env["SB_ROW_SHARD"])
            def shard(a):
                return a.take_rows(np.arange(g, len(a), G)[:len(a) // G])
            train_x, train_y, train_w = shard(train_x), shard(train_y), shard(train_w)
            valid_x, valid_y, valid_w = shard(valid_x), shard(valid_y), shard(valid_w)
    else:
        train_x = np.asarray(context["train_data"], dtype=np.float32)
        if train_x.ndim != 2 or train_x.shape[1] != feature_count:
            raise ValueError("training rows do not all have %d parsable features" % feature_count)
        train_y = np.asarray(context["train_target"], dtype=np.float32).reshape(-1)
        train_w = np.asarray(context["train_data_sample_weight"], dtype=np.float32).reshape(-1)
        valid_x = np.asarray(context["valid_data"], dtype=np.float32).reshape(-1, feature_count)
        valid_y = np.asarray(context["valid_target"], dtype=np.float32).reshape(-1)
        valid_w = np.asarray(context["valid_data_sample_weight"], dtype=np.float32).reshape(-1)
        if env.get("SB_ROW_SHARD"):
            # launcher.py: every local rank of a container reads the container's files and keeps rows g::G, cut to the
            # same length on every rank so that all ranks run the same number of exchanges
            train_x, train_y, train_w = row_shard(env["SB_ROW_SHARD"], train_x, train_y, train_w)
            valid_x, valid_y, valid_w = row_shard(env["SB_ROW_SHARD"], valid_x, valid_y, valid_w)
    vocab = offsets = None
    if wide_deep:
        # category codes -> global one-hot column indices.  V_c = SB_CATEGORY_VOCAB (space separated) or max code + 1 over the
        # data this rank sees (several ranks: set SB_CATEGORY_VOCAB so that every rank builds the same model)
        to_np = lambda a: a.numpy() if isinstance(a, capi.DeviceArray) else np.asarray(a, np.float32)
        train_x, train_y, train_w = to_np(train_x), to_np(train_y).reshape(-1), to_np(train_w).reshape(-1)
        valid_x, valid_y, valid_w = to_np(valid_x).reshape(-1, feature_count), to_np(valid_y).reshape(-1), to_np(valid_w).reshape(-1)
        n_dense, n_cat = len(numeric_cols), len(category_cols)
        codes = lambda X: np.where((X[:, n_dense:] >= 0) & (X[:, n_dense:] == np.floor(X[:, n_dense:])), X[:, n_dense:], -1).astype(np.int64)
        tr_codes, va_codes = codes(train_x), codes(valid_x)
        if env.get("SB_CATEGORY_VOCAB"):
            vocab = [int(v) for v in env["SB_CATEGORY_VOCAB"].split()]
            if len(vocab) != n_cat:
                raise ValueError("SB_CATEGORY_VOCAB must list %d sizes" % n_cat)
        else:
            if n_workers > 1:
                raise ValueError("wide+deep with several workers needs SB_CATEGORY_VOCAB (every rank must build the same model)")
            vocab = [int(max(1, tr_codes[:, c].max(initial=-1) + 1, va_codes[:, c].max(initial=-1) + 1)) for c in range(n_cat)]
        offsets = np.concatenate([[0], np.cumsum(vocab)[:-1]]).astype(np.int64)

        def to_idx(cd):
            ok = (cd >= 0) & (cd < np.asarray(vocab)[None, :])
            return np.where(ok, cd + offsets[None, :], -1).astype(np.int32)
        train_idx, valid_idx = to_idx(tr_codes), to_idx(va_codes)
        train_x, valid_x = np.ascontiguousarray(train_x[:, :n_dense]), np.ascontiguousarray(valid_x[:, :n_dense])
        feature_count = n_dense + int(sum(vocab))
        logging.info("wide+deep: %d dense + %d one-hot columns (%d categorical, vocabularies %s)" % (n_dense, sum(vocab), n_cat, vocab))
    logging.info("Testing set size: %d" % len(valid_x))
    logging.info("Training set size: %d" % len(train_x))

    # split data into batch (ssgd_monitor.py:189-192): int(N / BATCH_SIZE) near-equal batches
    total_batch = max(1, int(len(train_x) / batch_size))
    bounds = [b[0] for b in np.array_split(np.arange(len(train_x)), total_batch)] + [len(train_x)]
    max_rows = max(bounds[i + 1] - bounds[i] for i in range(total_batch))

    desc = model(feature_count, model_conf, max_rows)
    rdv = Rendezvous(cluster_spec, task_index, n_workers)
    nccl_id = exchange_nccl_id(rdv)
    trainer = capi.Trainer(desc, device=device, nccl_id=nccl_id, rank=task_index, world=n_workers)
    if n_workers > 1 and env.get("SB_EXCHANGE", "p2p") != "nccl":
        if enable_peer_exchange(trainer, rdv):
            logging.info("gradient exchange: peer-memory kernels (all %d ranks on this host)" % n_workers)
    # The reference has ONE copy of the variables (on the parameter servers); the chief alone initialises or restores it
    # (MonitoredTrainingSession(is_chief=...), ssgd_monitor.py:251-257).  Replicas: worker 0 initialises / restores, then
    # parameters, optimizer state and global_step are broadcast, so every rank starts from the same state and runs the
    # same number of exchanges even when only worker 0 can see the checkpoint.
    remote_tmp = _Fs.is_remote(tmp_model_path)
    ckpt_dir = tempfile.mkdtemp(prefix="sb_ckpt_") if remote_tmp else _Fs.local(tmp_model_path)
    ckpt = os.path.join(ckpt_dir, "model.ckpt")
    if is_chief or n_workers == 1:
        if remote_tmp and _Fs.exists(tmp_model_path.rstrip("/") + "/model.ckpt"):
            _Fs.fetch(tmp_model_path.rstrip("/") + "/model.ckpt", ckpt)
        if os.path.exists(ckpt):                  # MonitoredTrainingSession restores the latest checkpoint (:251-257)
            trainer.load_checkpoint(ckpt)
        else:
            trainer.init_xavier(int(env.get("SB_SEED", "0")) or random.SystemRandom().randrange(1, 2 ** 31))
    if n_workers > 1:
        trainer.broadcast_state(0)
    rdv.close()
    if wide_deep:
        trainer.set_sparse(len(numeric_cols), int(sum(vocab)), len(category_cols))
        if not per_batch_update:
            logging.info("wide+deep trains with one update per mini-batch (Schedule=batch); the sync-replicas accumulator is not wired for sparse steps")
            per_batch_update = True
        trainer.load_dataset_sparse(train_x, train_idx, train_y, train_w)
    else:
        trainer.load_dataset(train_x, train_y, train_w)

    # replicas_to_aggregate (ssgd_monitor.py:139): accepted pushes per global update, over all workers
    R = max(1, int(total_training_data_number * (1 - valid_ratio) / batch_size * REPLICAS_TO_AGGREGATE_RATIO))
    sched = SyncReplicasSchedule(R, n_workers)
    sched.global_step = trainer.global_step       # a restored run continues from the checkpoint's step (tokens restart at it)
    sched.local_step = [sched.global_step] * n_workers
    sched.tokens = [sched.global_step] * sched.R

    logging.info('Starting training on worker %d' % task_index)
    while trainer.global_step < epochs:           # StopAtStepHook(num_steps=EPOCH) (ssgd_monitor.py:235)
        start = time.time()
        l = 0.0
        if per_batch_update:
            # the whole `for i in range(total_batch): sess.run(train_step)` loop (ssgd_monitor.py:272-276) as one
            # asynchronous call per run of equally sized batches (np.array_split sizes differ by at most one row)
            for first, count, rows in equal_size_runs(bounds):
                n = min(count, epochs - trainer.global_step)
                if n <= 0:
                    break
                trainer.run_resident([int(b) for b in bounds[first:first + n]], rows)
            l = trainer.last_loss()
        else:
            i = 0
            while i < total_batch:
                ran, accepted, apply_now, pushes = sched.round()
                if ran[task_index]:
                    off, rows = int(bounds[i]), int(bounds[i + 1] - bounds[i])
                    if accepted[task_index]:
                        l = trainer.accumulate_resident(off, rows)
                    else:
                        l = trainer.loss_resident(off, rows)     # stale push: the run still reports its loss (:276)
                    i += 1
                if apply_now:
                    trainer.apply_accumulated(pushes)
                if trainer.global_step >= epochs:
                    break
        training_time = time.time() - start
        if wide_deep:
            valid_loss = trainer.eval_loss_sparse(valid_x, valid_idx, valid_y, valid_w) if len(valid_x) else 0.0
        else:
            valid_loss = trainer.eval_loss(valid_x, valid_y, valid_w) if len(valid_x) else 0.0
        gs = trainer.global_step
        logging.info('Step: ' + str(gs) + ' worker: ' + str(task_index) + " training loss:" + str(l) +
                     " valid loss:" + str(valid_loss))
        message = "worker_index:{},time:{},current_epoch:{},training_loss:{},valid_loss:{}\n".format(
            str(task_index), str(training_time), str(gs), str(l), str(valid_loss))
        if socket_client is not None:
            socket_client.send(message.encode('utf8'))
        if is_chief:
            os.makedirs(ckpt_dir, exist_ok=True)
            trainer.save_checkpoint(ckpt)
            if remote_tmp:
                _Fs.upload(ckpt, tmp_model_path.rstrip("/") + "/model.ckpt")

    logging.info('Done' + str(task_index))
    if is_chief:
        logging.info("Exporting saved_model to: {}".format(final_model_path))
        simple_save(trainer, final_model_path)
        logging.info("Exported saved_model")
    if n_workers > 1:
        # the chief's export / last checkpoint pull every rank's share of the fp32 master over peer memory: nobody frees
        # its arena before the chief is done (an all-reduce of nothing on the trainers' own communicator is the barrier)
        trainer.broadcast_state(0)
    trainer.close()
    if socket_client is not None:
        socket_client.close()
    logging.info('Session from worker %d closed cleanly' % task_index)
    return 0


if __name__ == '__main__':
    sys.exit(main())
