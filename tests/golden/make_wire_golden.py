"""Record lm:// wire transcripts against the reference's own server and client (LMCache v0.1.2).

    python tests/golden/make_wire_golden.py <path to the LMCache v0.1.2 source tree>

Output (committed): tests/golden/golden_wire.json.  A recording proxy sits between a client and the reference's
`python -m lmcache.server` (lmcache/server/__main__.py:29-104) and logs every frame in order:
  * "our_clients"       this package's lm:// and lmn:// clients running the session of
                        tests/test_c4_flow_cpu.py::_our_client_session -- the bytes they sent and the reference server's
                        replies.  Both clients must send the same bytes, so one transcript serves both.
  * "reference_client"  the reference's LMCServerConnector (lmcache/storage_backend/connector/lm_connector.py:15-84)
                        running _reference_client_session below -- its requests and the reference server's replies.
A frame is {"from": "client"|"server", ...} with "hex" (a header, verbatim), "blob" (a PUT / GET payload: index into the
session's blobs, which the tests regenerate) or "keys" (a LIST payload, in the reference server's order).
"""
import json
import os
import socket
import struct
import subprocess
import sys
import threading
import time

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
CLIENT_HDR, SERVER_HDR = 158, 8          # struct "ii150s" / "ii" (lmcache/protocol.py:30-70)
PUT, GET, LIST = 1, 2, 4


def _recv_exact(s, n):
    buf = bytearray()
    while len(buf) < n:
        k = s.recv(n - len(buf))
        if not k:
            return None
        buf += k
    return bytes(buf)


def _label(data, blobs, keys_payload):
    if keys_payload:
        return {"keys": data.decode().split("\n") if data else []}
    for i, b in enumerate(blobs):
        if data == b:
            return {"blob": i}
    return {"hex": data.hex()}


class RecordingProxy:
    """Accepts ONE client connection, forwards it to `upstream`, logs the frames of the exchange."""

    def __init__(self, upstream_port, blobs):
        self.lsock = socket.socket()
        self.lsock.bind(("127.0.0.1", 0))
        self.lsock.listen(1)
        self.port = self.lsock.getsockname()[1]
        self.upstream_port, self.blobs, self.frames = upstream_port, list(blobs), []
        self.thread = threading.Thread(target=self._run)
        self.thread.start()

    def _run(self):
        cli, _ = self.lsock.accept()
        up = socket.create_connection(("127.0.0.1", self.upstream_port))
        while True:
            hdr = _recv_exact(cli, CLIENT_HDR)
            if hdr is None:
                break
            self.frames.append({"from": "client", "hex": hdr.hex()})
            up.sendall(hdr)
            cmd, length = struct.unpack("ii", hdr[:8])
            if cmd == PUT:
                payload = _recv_exact(cli, length)
                self.frames.append(dict({"from": "client"}, **_label(payload, self.blobs, False)))
                up.sendall(payload)
                continue
            rep = _recv_exact(up, SERVER_HDR)
            self.frames.append({"from": "server", "hex": rep.hex()})
            cli.sendall(rep)
            code, n = struct.unpack("ii", rep)
            if cmd in (GET, LIST) and code == 200:
                data = _recv_exact(up, n)
                self.frames.append(dict({"from": "server"}, **_label(data, self.blobs, cmd == LIST)))
                cli.sendall(data)
        up.close()
        cli.close()
        self.lsock.close()

    def transcript(self):
        self.thread.join()
        return self.frames


def _reference_client_session(c, blobs):
    """What the reference's own client does against an lm:// server (formerly run in a subprocess by
    tests/test_c4_flow_cpu.py::test_reference_client_against_our_native_server)."""
    for k, v in blobs.items():
        c.set(k, v)
    for k, v in blobs.items():
        for _ in range(400):
            if c.exists(k):
                break
            time.sleep(0.005)
        assert c.exists(k) and bytes(c.get(k)) == v, k
    assert not c.exists("nope@x@1@0@00") and c.get("nope@x@1@0@00") is None
    assert sorted(c.list()) == sorted(blobs)
    c.close()


def _with_reference_server(ref, fn):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(TESTS, "_refstubs"), ref]))
    srv = subprocess.Popen([sys.executable, "-m", "lmcache.server", "127.0.0.1", str(port)], env=env, cwd=ref,
                           stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    try:
        for _ in range(900):
            try:
                socket.create_connection(("127.0.0.1", port), timeout=0.2).close()
                break
            except OSError:
                assert srv.poll() is None, "reference server exited"
                time.sleep(0.1)
        return fn(port)
    finally:
        srv.terminate()
        srv.wait()


def main():
    ref = os.path.abspath(sys.argv[1])
    sys.path[:0] = [ROOT, TESTS, os.path.join(TESTS, "_refstubs"), ref]
    import __graft_entry__ as ge
    ge.build_cuda()
    import test_c4_flow_cpu as T
    from lmcache.storage_backend.connector.lm_connector import LMCServerConnector as RefConnector

    from lmcache_b200.storage_backend.connector import CreateConnector

    out = {}
    ours = {}
    for scheme in ("lm", "lmn"):
        def run(port):
            blobs = T._our_client_blobs()
            px = RecordingProxy(port, blobs.values())
            T._our_client_session(CreateConnector(f"{scheme}://127.0.0.1:{px.port}"), blobs)
            return px.transcript()
        ours[scheme] = _with_reference_server(ref, run)
    assert ours["lm"] == ours["lmn"], "the lm:// and lmn:// clients sent different bytes"
    out["our_clients"] = ours["lm"]

    def run_ref(port):
        blobs = T._reference_client_blobs()
        px = RecordingProxy(port, blobs.values())
        _reference_client_session(RefConnector("127.0.0.1", px.port), blobs)
        return px.transcript()
    out["reference_client"] = _with_reference_server(ref, run_ref)
    with open(os.path.join(HERE, "golden_wire.json"), "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    print({k: len(v) for k, v in out.items()}, "frames written")


if __name__ == "__main__":
    main()
