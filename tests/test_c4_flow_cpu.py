"""CPU: (1) the BASELINE configs[3] flow across processes -- a writer process, a reader process and one lm:// server
process -- at the level that needs no GPU: token ids -> SHA-256 chain -> engine key strings -> B2KV containers over the
wire -> header checks -> decode, with the CPU oracle standing in for the kernels on both sides;
(2) wire interoperability with the REFERENCE's own server and client (lmcache/server/__main__.py:29-104,
lmcache/storage_backend/connector/lm_connector.py:15-84), through sessions recorded against them
(tests/golden/golden_wire.json, made by tests/golden/make_wire_golden.py)."""
import ctypes
import json
import os
import socket
import subprocess
import sys
import threading
import time

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _wait_port(port, proc=None, tries=900):
    for _ in range(tries):
        try:
            socket.create_connection(("127.0.0.1", port), timeout=0.2).close()
            return True
        except OSError:
            if proc is not None and proc.poll() is not None:
                return False
            time.sleep(0.1)
    return False


WORKER = r'''
import os, sys, json
import numpy as np
sys.path.insert(0, {root!r})
import torch
from oracle import oracle as O
from lmcache_b200.codec import parse_header
from lmcache_b200.storage_backend.connector import CreateConnector
from lmcache_b200.storage_backend.serde.cachegen_basics import CacheGenGPUBytestream, CacheGenGPUEncoderOutput
from lmcache_b200.utils import CacheEngineKey
role, url, coder = sys.argv[1], sys.argv[2], int(sys.argv[3])
MODEL, L, H, D, T, cs = "lmsys/longchat-7b-16k", 3, 2, 16, 600, 256
tokens = np.random.default_rng(42).integers(0, 32000, T, dtype=np.int64)
bits = O.synth_kv_bits(L, T, H * D, seed=9)
kb, vb = O.make_bins(MODEL)
keys = [CacheEngineKey("vllm", MODEL, 2, 0, h).to_string() for h in O.sha256_chain(tokens, cs)]
conn = CreateConnector(url)
if role == "writer":
    for j, key in enumerate(keys):
        x = bits[:, :, j * cs:(j + 1) * cs]
        t = x.shape[2]
        enc = O.encode_chunk(x, O.DT_BF16, kb, vb, coder)
        mk = torch.from_numpy(enc["maxes"][0].view(np.int16)).view(torch.bfloat16).reshape(L, t, 1)
        mv = torch.from_numpy(enc["maxes"][1].view(np.int16)).view(torch.bfloat16).reshape(L, t, 1)
        raw = CacheGenGPUEncoderOutput([CacheGenGPUBytestream(torch.from_numpy(b), torch.from_numpy(ln), g) for b, ln, g in enc["groups"]],
                                       torch.from_numpy(enc["cdf"]), mk, mv, H, D, coder,
                                       torch.from_numpy(O.counts(enc["sym"]).astype(np.int32)), O.nb_map(kb, vb, L)).to_bytes()
        assert raw[4] == coder + 1
        conn.set(key, raw)
    assert conn.exists(keys[-1]) or True          # one round trip: the server has consumed the PUTs before it
    print(json.dumps({{"stored": len(keys)}}))
else:
    got, ok = 0, True
    for j, key in enumerate(keys + [CacheEngineKey("vllm", MODEL, 2, 0, "0" * 64).to_string()]):
        bs = conn.get(key)
        if bs is None:
            break
        hd = parse_header(bs)                     # structural checks of the flat container
        out = CacheGenGPUEncoderOutput.from_bytes(bytes(bs))
        enc = dict(cdf=out.cdf.numpy(), maxes=np.stack([out.max_tensors_key.view(torch.int16).numpy().view(np.uint16).reshape(L, -1),
                                                         out.max_tensors_value.view(torch.int16).numpy().view(np.uint16).reshape(L, -1)]),
                   groups=[(c.bytestream.numpy(), c.bytestream_lengths.numpy(), c.ntokens) for c in out.data_chunks], coder=out.coder)
        dec = O.decode_chunk(enc, O.DT_BF16, kb, vb, O.DT_BF16)
        x = bits[:, :, j * cs:(j + 1) * cs]
        want = O.decode_chunk(O.encode_chunk(x, O.DT_BF16, kb, vb, coder), O.DT_BF16, kb, vb, O.DT_BF16)
        ok = ok and hd.ntokens == x.shape[2] and np.array_equal(dec, want)
        got += 1
    print(json.dumps({{"hits": got, "ok": bool(ok)}}))
conn.close()
'''


@pytest.mark.parametrize("coder", [0, 1, 2])
@pytest.mark.parametrize("server_kind", ["native", "python"])
def test_c4_flow_two_processes_one_server(coder, server_kind, tmp_path):
    import json
    port = _free_port()
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    args = [sys.executable, "-m", "lmcache_b200.server", "127.0.0.1", str(port)] + (["--python"] if server_kind == "python" else [])
    srv = subprocess.Popen(args, env=env)
    try:
        assert _wait_port(port, srv)
        script = tmp_path / "worker.py"
        script.write_text(WORKER.format(root=ROOT))
        url = f"lm://127.0.0.1:{port}"
        w = subprocess.run([sys.executable, str(script), "writer", url, str(coder)], env=env, capture_output=True, text=True, timeout=300)
        assert w.returncode == 0, w.stderr[-2000:]
        assert json.loads(w.stdout.strip().splitlines()[-1]) == {"stored": 3}
        r = subprocess.run([sys.executable, str(script), "reader", url.replace("lm://", "lmn://"), str(coder)], env=env,
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1]) == {"hits": 3, "ok": True}     # 2 full chunks + the 88-token tail, then a miss
    finally:
        srv.terminate()
        srv.wait()


def _our_client_blobs():
    rng = np.random.default_rng(5)
    return {f"vllm@lmsys/longchat-7b-16k@2@0@{i:064x}": rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            for i, n in enumerate([1, 157, 65536, 2 * 1024 * 1024 + 3])}


def _reference_client_blobs():
    return {"vllm@a/b@1@0@" + "%064x" % i: bytes([i]) * n for i, n in enumerate([1, 158, 70000, 1 << 21])}


def _our_client_session(c, blobs):
    """set / exists / get / get_into / miss / list through one of this package's clients (also what
    tests/golden/make_wire_golden.py ran against the reference server)"""
    for k, v in blobs.items():
        c.set(k, v)
    for k, v in blobs.items():
        for _ in range(400):
            if c.exists(k):
                break
            time.sleep(0.005)
        assert c.exists(k)
        assert bytes(c.get(k)) == v
        buf = np.zeros(len(v) + 64, np.uint8)
        assert c.get_into(k, buf.ctypes.data, buf.size) == len(v) and buf[:len(v)].tobytes() == v
    assert not c.exists("vllm@m@1@0@" + "f" * 64) and c.get("vllm@m@1@0@" + "f" * 64) is None
    assert sorted(c.list()) == sorted(blobs)
    c.close()


def _transcript(name):
    """frames of a session recorded against the reference's own server (tests/golden/make_wire_golden.py)"""
    return json.load(open(os.path.join(HERE, "golden", "golden_wire.json")))[name]


def _frame_bytes(f, blobs):
    if "hex" in f:
        return bytes.fromhex(f["hex"])
    if "blob" in f:
        return blobs[f["blob"]]
    return "\n".join(f["keys"]).encode()


def _recv_exact(s, n):
    buf = bytearray()
    while len(buf) < n:
        k = s.recv(n - len(buf))
        if not k:
            raise AssertionError(f"connection closed after {len(buf)} of {n} bytes")
        buf += k
    return bytes(buf)


class _ReferenceServerReplay:
    """Plays the reference server's side of a recorded session to ONE client: every byte the client sends must be the
    byte the reference server received, and the client gets the reference server's replies verbatim."""

    def __init__(self, frames, blobs):
        self.lsock = socket.socket()
        self.lsock.bind(("127.0.0.1", 0))
        self.lsock.listen(1)
        self.lsock.settimeout(60)
        self.port = self.lsock.getsockname()[1]
        self.frames, self.blobs, self.error = frames, blobs, None
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        try:
            cli, _ = self.lsock.accept()
            cli.settimeout(60)
            with cli:
                for i, f in enumerate(self.frames):
                    want = _frame_bytes(f, self.blobs)
                    if f["from"] == "server":
                        cli.sendall(want)
                    else:
                        got = _recv_exact(cli, len(want))
                        assert got == want, f"frame {i}: the client sent {got[:200]!r}, the reference server received {want[:200]!r}"
                assert cli.recv(1) == b"", "the client sent more than the recorded session"
        except BaseException as e:       # noqa: BLE001 -- reported by join() on the test's thread
            self.error = e
        finally:
            self.lsock.close()

    def join(self):
        self.thread.join(120)
        assert not self.thread.is_alive(), "replay server still waiting for the client"
        if self.error is not None:
            raise self.error


@pytest.mark.parametrize("scheme", ["lm", "lmn"])
def test_our_clients_against_the_reference_server(scheme):
    """This package's two lm:// clients against the reference's `python -m lmcache.server`, replayed from a recorded
    session: requests byte-identical to what that server accepted, its replies understood."""
    from lmcache_b200.storage_backend.connector import CreateConnector
    blobs = _our_client_blobs()
    srv = _ReferenceServerReplay(_transcript("our_clients"), list(blobs.values()))
    try:
        _our_client_session(CreateConnector(f"{scheme}://127.0.0.1:{srv.port}"), blobs)
    finally:
        srv.join()


def test_reference_client_against_our_native_server():
    """The reference's LMCServerConnector against csrc/lmnet.cu's server: the requests that client sent in a recorded
    session go to our server, whose replies must be the reference server's (LIST: the same keys, in any order)."""
    import __graft_entry__ as ge
    ge.build_cuda()
    from lmcache_b200 import _native as N
    lib = N.lib()
    h = ctypes.c_void_p()
    N.check(lib.b200kv_lm_server_start(b"127.0.0.1", 0, ctypes.byref(h)))
    port = lib.b200kv_lm_server_port(h)
    blobs = list(_reference_client_blobs().values())
    try:
        with socket.create_connection(("127.0.0.1", port), timeout=60) as s:
            for i, f in enumerate(_transcript("reference_client")):
                want = _frame_bytes(f, blobs)
                if f["from"] == "client":
                    s.sendall(want)
                    continue
                got = _recv_exact(s, len(want))
                if "keys" in f:
                    assert sorted(got.decode().split("\n")) == sorted(f["keys"]), f"frame {i}: LIST"
                else:
                    assert got == want, f"frame {i}: our server replied {got[:200]!r}, the reference server {want[:200]!r}"
        assert lib.b200kv_lm_server_num_keys(h) == 4
    finally:
        N.check(lib.b200kv_lm_server_stop(h))
