"""Mesh runtime: ``P2PNode`` + ``run_p2p_node`` (parity: /root/reference/bee2bee/p2p_runtime.py).

Same public surface and wire messages as the reference (hello / peer_list / ping / pong /
service_announce / gen_request / gen_chunk / gen_success / gen_error / gen_result /
piece_request / piece_data, section 2.5 of SURVEY.md), re-designed:

* transports are pluggable (``ws://`` wire-compatible sockets, ``inproc://`` hub) and carry
  only the *control plane*; activations between layer pieces move GPU->GPU (``parallel.mesh``)
  or, on CPU-only hosts, as binary ``hidden_forward`` frames -- never JSON number lists;
* handlers never block the loop: services run through ``aexecute`` / ``aexecute_stream``;
* a requester resolves on ``gen_success | gen_error | gen_result`` and streams ``gen_chunk``
  (the reference only resolves ``gen_result`` and times out, SURVEY R8);
* failure detection: missed pongs mark a peer unreachable and drop it; bootstrap peers are
  re-dialled with back-off; byte-piece exchange and the DHT are actually wired.
"""
from __future__ import annotations

import asyncio
import base64
import json
import os
import time
from typing import Any, Awaitable, Callable, Dict, List, Optional, Tuple

from . import protocol as P
from .dht import DHTNode, announce_piece
from .p2p import generate_join_link, parse_join_link, registration_url, sha256_hex_bytes
from .pieces import LayerPiece, piece_hashes, split_pieces, verify_and_reassemble
from .registry import RegistryClient
from .services import BaseService, ServiceError, build_service
from .transport import Connection, ConnectionClosed, InProcHub, WSServer, connect, ws_listen
from .utils import get_lan_ip, get_public_ip, get_system_metrics, new_id, now_ms, offline, sha256_hex

try:
    from loguru import logger
except Exception:  # pragma: no cover
    import logging

    logger = logging.getLogger("bee2bee")

DEFAULT_GEN_TIMEOUT = 300.0          # reference: p2p_runtime.py:831
BLOB_PIECE_SIZE = 1 << 20


class P2PNode:
    def __init__(self, host: str = "0.0.0.0", port: int = 4001, announce_host: Optional[str] = None,
                 announce_port: Optional[int] = None, entrypoint_url: Optional[str] = None, region: str = "Auto",
                 transport: str = "ws", name: Optional[str] = None, health_interval: float = 15.0,
                 pong_timeout: float = 45.0):
        self.host, self.port = host, port
        self.announce_host, self.announce_port = announce_host, announce_port
        self.peer_id = new_id("peer")
        self.registry = RegistryClient(entrypoint_url=entrypoint_url)
        self.region = region
        self.transport = transport                       # "ws" | "inproc"
        self.name = name or self.peer_id
        self.addr = ""
        self.server: Optional[WSServer] = None
        self.public_ip: Optional[str] = None
        self.api_port: Optional[int] = None
        self.api_host: Optional[str] = None
        self.start_time: Optional[float] = None
        # ---- state
        self.peers: Dict[str, Dict[str, Any]] = {}          # pid -> {ws, addr, last_pong_ms, metrics, ...}
        self.local_services: Dict[str, BaseService] = {}
        self.providers: Dict[str, Dict[str, Any]] = {}      # pid -> {svc_name: meta, "_latency": ms}
        self.pieces: Dict[str, Dict[str, Any]] = {}         # content_hash -> {hashes, size, chunks}
        self.layer_pieces: List[LayerPiece] = []            # layer ranges hosted here
        self.remote_layer_pieces: Dict[str, List[Dict[str, Any]]] = {}
        self.piece_hosts: Dict[str, Any] = {}               # "model:index" -> PieceHost (CPU pipeline hop)
        self.dht = DHTNode(mesh_local=True)
        self._lock = asyncio.Lock()
        self._pending_requests: Dict[str, asyncio.Future] = {}
        self._stream_sinks: Dict[str, Callable[[str], None]] = {}
        self._pending_blobs: Dict[str, Dict[str, Any]] = {}
        self._pending_hidden: Dict[str, asyncio.Future] = {}
        self._bootstrap_addrs: List[str] = []
        self._tasks: List[asyncio.Task] = []
        self._running = False
        self._monitor_active = False
        self.health_interval, self.pong_timeout = health_interval, pong_timeout
        self._handlers: Dict[str, Callable[[Connection, Dict[str, Any]], Awaitable[None]]] = {
            P.HELLO: self._handle_hello, P.PEER_LIST: self._handle_peer_list, P.PING: self._handle_ping,
            P.PONG: self._handle_pong, P.SERVICE_ANNOUNCE: self._handle_service_announce,
            P.GEN_REQUEST: self._handle_gen_request, P.GEN_CHUNK: self._handle_gen_chunk,
            P.GEN_SUCCESS: self._handle_gen_terminal, P.GEN_ERROR: self._handle_gen_terminal,
            P.GEN_RESULT: self._handle_gen_terminal, P.PIECE_REQUEST: self._handle_piece_request,
            P.PIECE_DATA: self._handle_piece_data, P.PIECE_ANNOUNCE: self._handle_piece_announce,
            P.HIDDEN_FORWARD: self._handle_hidden_forward, P.HIDDEN_RESULT: self._handle_hidden_result,
        }

    # =============================================================== lifecycle
    async def start(self) -> None:
        if self._running:
            return
        self._running = True
        self.start_time = time.time()
        await self.dht.start()
        if self.transport == "inproc" or self.host.startswith("inproc"):
            self.addr = InProcHub.listen(self.name, self._on_incoming)
        else:
            self.server = await ws_listen(self.host, self.port, self._on_incoming)
            self.port = self.server.port
            host = self.announce_host
            if not host:
                host = get_lan_ip() if self.host in ("0.0.0.0", "", "::") else self.host
                if self.host in ("0.0.0.0", "", "::") and not offline():
                    await self._try_nat()
            self.addr = f"ws://{host}:{self.announce_port or self.port}"
        self._monitor_active = True
        self._tasks.append(asyncio.create_task(self._monitoring_loop(self.health_interval)))
        logger.info(f"P2P node {self.peer_id} listening at {self.addr}")

    async def _try_nat(self) -> None:
        """Best-effort public reachability (UPnP -> NAT-PMP -> PCP -> STUN); inert offline."""
        try:
            from .nat import auto_port_forward

            res = await asyncio.wait_for(auto_port_forward(self.port), timeout=8)
            if res and res.success and res.external_ip:
                self.public_ip = res.external_ip
                return
        except Exception as exc:
            logger.debug(f"NAT traversal skipped: {exc}")
        try:
            self.public_ip = await asyncio.get_running_loop().run_in_executor(None, get_public_ip)
        except Exception:
            self.public_ip = None

    async def stop(self) -> None:
        self._running = False
        self._monitor_active = False
        for t in self._tasks:
            t.cancel()
        self._tasks.clear()
        async with self._lock:
            conns = [p.get("ws") for p in self.peers.values()]
            self.peers.clear()
            self.providers.clear()
        for c in conns:
            if c is not None:
                try:
                    await c.close()
                except Exception:
                    pass
        if self.server is not None:
            await self.server.close()
            self.server = None
        if self.addr.startswith("inproc://"):
            InProcHub.unlisten(self.name)
        for fut in list(self._pending_requests.values()) + list(self._pending_hidden.values()):
            if not fut.done():
                fut.set_exception(ConnectionError("node stopped"))
        await self.dht.stop()

    async def enable_monitoring(self, interval_seconds: float = 30) -> None:
        """(Re)configure the supervisor loop.  Unlike the reference this is effective after
        ``start()`` too (there the flag is already set and the call is a no-op)."""
        self.health_interval = float(interval_seconds)
        if not self._monitor_active and self._running:
            self._monitor_active = True
            self._tasks.append(asyncio.create_task(self._monitoring_loop(self.health_interval)))

    async def _monitoring_loop(self, interval: float) -> None:
        while self._monitor_active and self._running:
            await asyncio.sleep(self.health_interval if self.health_interval else interval)
            try:
                await self._run_health_checks()
                if self.registry.enabled:
                    await self.sync_with_registry()
                await self._redial_bootstrap()
            except asyncio.CancelledError:
                raise
            except Exception as exc:
                logger.error(f"Monitoring error: {exc}")

    async def _refresh_local_services(self) -> None:
        """A local service whose engine lost its GPU mesh announces itself unhealthy: peers (and we) sort it last."""
        mine = self.providers.setdefault(self.peer_id, {})
        changed = []
        for name, svc in list(self.local_services.items()):
            try:
                meta = svc.get_metadata()
            except Exception:
                continue
            was = (mine.get(name) or {}).get("healthy", True)
            mine[name] = meta
            if meta.get("healthy", True) != was:
                logger.warning(f"service '{name}' is now {'healthy' if meta.get('healthy', True) else 'UNHEALTHY (GPU mesh aborted)'}")
                changed.append((name, meta))
        mine["health"] = "good" if all((m or {}).get("healthy", True) for k, m in mine.items()
                                       if not k.startswith("_") and isinstance(m, dict)) else "degraded"
        # our own view is settled before peers hear of the change: a peer that acts on the announce must not find this
        # node still preferring the service it just declared unhealthy
        for name, meta in changed:
            await self._broadcast(P.service_announce(name, meta))

    async def _run_health_checks(self) -> None:
        await self._refresh_local_services()
        metrics = get_system_metrics()
        stamp = now_ms()
        dead: List[str] = []
        for pid, info in list(self.peers.items()):
            conn: Optional[Connection] = info.get("ws")
            if conn is None or conn.closed:
                dead.append(pid)
                continue
            last = info.get("last_pong_at") or info.get("connected_at") or time.time()
            if time.time() - last > self.pong_timeout:
                info["health_status"] = "unreachable"
                if pid in self.providers:
                    self.providers[pid]["health"] = "degraded"
                dead.append(pid)
                continue
            ok = await self._send(conn, P.ping(metrics))
            info["last_audit"] = stamp
            info["health_status"] = "online" if ok else "unreachable"
            if pid in self.providers:
                self.providers[pid]["last_audit"] = stamp
                self.providers[pid]["health"] = "good" if ok else "degraded"
            if not ok:
                dead.append(pid)
        for pid in dead:
            await self._drop_peer(pid)

    async def _redial_bootstrap(self) -> None:
        known = {p.get("addr") for p in self.peers.values()}
        for addr in self._bootstrap_addrs:
            if addr not in known and addr != self.addr:
                try:
                    await self._connect_peer(addr)
                except Exception:
                    pass

    async def sync_with_registry(self) -> bool:
        if not self.addr:
            return False
        metrics = get_system_metrics()
        metrics["api_port"] = self.api_port or 8000
        metrics["backend"] = "b200-native"
        models: List[str] = []
        for svc in self.local_services.values():
            meta = svc.get_metadata()
            models.extend(meta.get("models") or ([meta["model"]] if "model" in meta else []))
        return await self.registry.sync_node(peer_id=self.peer_id, address=self.addr, models=sorted(set(models)),
                                             tag="b200-production", region=self.region, metrics=metrics)

    # ============================================================ connections
    async def connect_bootstrap(self, link: str) -> bool:
        """Join link (``coithub.org://``, ``coithub://``, ``p2pnet://``) or raw ws/inproc address."""
        addrs: List[str]
        if "://join?" in link:
            try:
                addrs = parse_join_link(link)["bootstrap"]
            except ValueError:
                logger.error(f"Invalid bootstrap link: {link}")
                return False
        else:
            addrs = [link]
        ok = False
        for a in addrs:
            if a not in self._bootstrap_addrs:
                self._bootstrap_addrs.append(a)
            try:
                await self._connect_peer(a)
                ok = True
            except Exception as exc:
                logger.warning(f"Bootstrap {a} unreachable: {exc}")
        return ok

    async def _connect_peer(self, addr: str) -> Optional[str]:
        if addr == self.addr or any(p.get("addr") == addr for p in self.peers.values()):
            return None
        conn = await connect(addr)
        tmp = new_id("tmp")
        async with self._lock:
            self.peers[tmp] = {"ws": conn, "addr": addr, "last_pong_ms": 0, "metrics": None,
                               "connected_at": time.time(), "health_status": "connecting"}
        await self._send(conn, self._make_hello_msg())
        self._tasks.append(asyncio.create_task(self._peer_reader(conn)))
        return tmp

    async def _on_incoming(self, conn: Connection) -> None:
        tmp = new_id("in")
        async with self._lock:
            self.peers[tmp] = {"ws": conn, "addr": None, "last_pong_ms": 0, "metrics": None,
                               "connected_at": time.time(), "health_status": "connecting"}
        await self._peer_reader(conn)

    async def _peer_reader(self, conn: Connection) -> None:
        try:
            async for raw in conn:
                try:
                    data = json.loads(raw)
                except ValueError:
                    continue
                if P.is_message(data):
                    await self._on_message(conn, data)
        except asyncio.CancelledError:
            raise
        except Exception as exc:
            logger.debug(f"peer reader ended: {exc}")
        finally:
            await self._on_disconnect(conn)

    async def _on_disconnect(self, conn: Connection) -> None:
        gone = [pid for pid, info in self.peers.items() if info.get("ws") is conn]
        for pid in gone:
            await self._drop_peer(pid, close=False)

    async def _drop_peer(self, pid: str, close: bool = True) -> None:
        async with self._lock:
            info = self.peers.pop(pid, None)
            self.providers.pop(pid, None)
            self.remote_layer_pieces.pop(pid, None)
        if info and close and info.get("ws") is not None:
            try:
                await info["ws"].close()
            except Exception:
                pass
        # fail requests that were waiting on this peer instead of letting them time out
        for rid, fut in list(self._pending_requests.items()):
            if getattr(fut, "_b2b_peer", None) == pid and not fut.done():
                fut.set_result({"error": f"relay_link_failure: peer {pid} disconnected"})

    async def _send(self, conn: Optional[Connection], message: Dict[str, Any]) -> bool:
        """Returns False on failure (the reference swallows send errors, which makes its
        "unreachable" health state unreachable -- SURVEY section 8)."""
        if conn is None:
            return False
        try:
            await conn.send(json.dumps(message))
            return True
        except (ConnectionClosed, Exception) as exc:
            logger.debug(f"send failed: {exc}")
            return False

    async def _broadcast(self, message: Dict[str, Any]) -> int:
        conns = [info.get("ws") for info in self.peers.values()]
        results = await asyncio.gather(*(self._send(c, message) for c in conns), return_exceptions=True)
        return sum(1 for r in results if r is True)

    def _conn_of(self, pid: str) -> Optional[Connection]:
        return (self.peers.get(pid) or {}).get("ws")

    def _pid_of(self, conn: Connection) -> Optional[str]:
        for pid, info in self.peers.items():
            if info.get("ws") is conn:
                return pid
        return None

    # ================================================================ services
    async def add_service(self, svc: BaseService) -> None:
        self.local_services[svc.name] = svc
        meta = svc.get_metadata()
        self.providers.setdefault(self.peer_id, {})[svc.name] = meta
        self.providers[self.peer_id]["_latency"] = 0.0
        for m in meta.get("models", []):
            await announce_piece(self.dht, "model:" + sha256_hex(m), self.addr or self.peer_id)
        await self._broadcast(P.service_announce(svc.name, meta))

    async def add_hf_service(self, model_name: str, price_per_token: float = 0.0, **kw) -> BaseService:
        svc = build_service("hf", model_name, price_per_token=price_per_token, **kw)
        await asyncio.get_running_loop().run_in_executor(None, svc.load_sync)
        await self.add_service(svc)
        return svc

    def add_layer_piece(self, piece: LayerPiece) -> None:
        piece.peer_id = self.peer_id
        self.layer_pieces.append(piece)

    def _make_hello_msg(self) -> Dict[str, Any]:
        services = {name: svc.get_metadata() for name, svc in self.local_services.items()}
        return P.hello(self.peer_id, self.addr, self.region, get_system_metrics(), services, api_port=self.api_port,
                       api_host=self.api_host, public_ip=self.public_ip,
                       pieces=[p.describe() for p in self.layer_pieces])

    # ================================================================ dispatch
    async def _on_message(self, conn: Connection, data: Dict[str, Any]) -> None:
        handler = self._handlers.get(data.get("type"))
        if handler is None:
            logger.debug(f"unknown message type {data.get('type')!r} dropped")
            return
        try:
            await handler(conn, data)
        except Exception as exc:
            logger.error(f"handler {data.get('type')} failed: {exc!r}")

    async def _handle_hello(self, conn: Connection, data: Dict[str, Any]) -> None:
        pid, addr = data.get("peer_id"), data.get("addr")
        if not pid or pid == self.peer_id:
            return
        first_contact = False
        async with self._lock:
            old = self._pid_of(conn)
            prev = self.peers.pop(old, {}) if old and old != pid else self.peers.get(pid, {})
            first_contact = not prev.get("hello_seen")
            entry = {"ws": conn, "addr": addr or prev.get("addr"), "last_pong_ms": prev.get("last_pong_ms", 0),
                     "metrics": data.get("metrics") or prev.get("metrics"), "region": data.get("region"),
                     "api_port": data.get("api_port"), "api_host": data.get("api_host"),
                     "public_ip": data.get("public_ip"), "connected_at": prev.get("connected_at", time.time()),
                     "last_pong_at": prev.get("last_pong_at"), "health_status": "online", "hello_seen": True}
            self.peers[pid] = entry
            if data.get("services"):
                lat = self.providers.get(pid, {}).get("_latency")
                self.providers[pid] = dict(data["services"])
                if lat is not None:
                    self.providers[pid]["_latency"] = lat
            if data.get("pieces"):
                self.remote_layer_pieces[pid] = list(data["pieces"])
        if first_contact:
            await self._send(conn, self._make_hello_msg())
            await self._send(conn, P.peer_list([v["addr"] for v in self.peers.values() if v.get("addr")]))
            await self._send(conn, P.ping())

    async def _handle_peer_list(self, conn: Connection, data: Dict[str, Any]) -> None:
        for addr in data.get("peers", []):
            if not addr or addr == self.addr or any(v.get("addr") == addr for v in self.peers.values()):
                continue
            self._tasks.append(asyncio.create_task(self._safe_connect(addr)))

    async def _safe_connect(self, addr: str) -> None:
        try:
            await self._connect_peer(addr)
        except Exception as exc:
            logger.debug(f"gossip dial {addr} failed: {exc}")

    async def _handle_ping(self, conn: Connection, data: Dict[str, Any]) -> None:
        pid = self._pid_of(conn)
        if pid and data.get("metrics"):
            self.peers[pid]["metrics"] = data["metrics"]
        await self._send(conn, P.pong(data.get("ts")))

    async def _handle_pong(self, conn: Connection, data: Dict[str, Any]) -> None:
        pid = self._pid_of(conn)
        if not pid:
            return
        try:
            rtt = max(0.0, (time.time() - float(data.get("ts"))) * 1000.0)
        except (TypeError, ValueError):
            return
        self.peers[pid]["last_pong_ms"] = rtt
        self.peers[pid]["last_pong_at"] = time.time()
        self.peers[pid]["health_status"] = "online"
        if pid in self.providers:
            self.providers[pid]["_latency"] = rtt

    async def _handle_service_announce(self, conn: Connection, data: Dict[str, Any]) -> None:
        pid = self._pid_of(conn)
        if pid and data.get("service"):
            self.providers.setdefault(pid, {})[data["service"]] = data.get("meta") or {}

    async def _handle_piece_announce(self, conn: Connection, data: Dict[str, Any]) -> None:
        pid = self._pid_of(conn)
        if pid:
            self.remote_layer_pieces[pid] = list(data.get("pieces") or [])

    # ------------------------------------------------------------- generation
    def _find_local_service(self, svc_name: Optional[str], model: Optional[str]) -> Optional[BaseService]:
        svc = self.local_services.get(svc_name) if svc_name else None
        if svc is not None and svc.serves(model):
            return svc
        for cand in self.local_services.values():
            if model and cand.serves(model):
                return cand
        return svc if (svc is not None and not model) else None

    async def _handle_gen_request(self, conn: Connection, data: Dict[str, Any]) -> None:
        rid = P.request_id_of(data) or new_id("req")
        model = data.get("model")
        params = {"prompt": data.get("prompt"),
                  "max_new_tokens": int(data.get("max_new_tokens") or data.get("max_tokens") or 2048),
                  "temperature": data.get("temperature", 0.7)}
        svc = self._find_local_service(data.get("svc", "hf"), model)
        if svc is not None:
            # run as a task so this peer's reader keeps draining pings / other requests
            self._tasks.append(asyncio.create_task(self._serve_local(conn, rid, svc, params, bool(data.get("stream")))))
            return
        picked = self.pick_provider(model) if model else None
        if picked is None or picked[0] == self.peer_id:
            await self._send(conn, P.msg(P.GEN_RESULT, rid=rid, error="consensus_deadlock: no_node_available"))
            return
        self._tasks.append(asyncio.create_task(self._relay(conn, rid, picked[0], params, model)))

    async def _serve_local(self, conn: Connection, rid: str, svc: BaseService, params: Dict[str, Any],
                           stream: bool) -> None:
        try:
            if stream:
                async for raw in svc.aexecute_stream(params):
                    text = raw
                    try:                                  # NDJSON services: unwrap {"text": ...}
                        obj = json.loads(raw)
                        if isinstance(obj, dict):
                            if obj.get("done"):
                                continue
                            if obj.get("status") == "error" or "error" in obj:
                                raise ServiceError(obj.get("message") or obj.get("error"))
                            text = obj.get("text", "")
                    except ValueError:
                        pass
                    if text:
                        await self._send(conn, P.msg(P.GEN_CHUNK, rid=rid, text=text))
                await self._send(conn, P.msg(P.GEN_SUCCESS, rid=rid, text="", backend="b200-native"))
            else:
                result = await svc.aexecute(params)
                await self._send(conn, P.msg(P.GEN_SUCCESS, rid=rid, **result))
        except Exception as exc:
            await self._send(conn, P.msg(P.GEN_ERROR, rid=rid, error=f"local_error: {exc}"))

    async def _relay(self, conn: Connection, rid: str, pid: str, params: Dict[str, Any], model: Optional[str]) -> None:
        try:
            res = await self.request_generation(pid, params["prompt"], params["max_new_tokens"], model,
                                                temperature=params.get("temperature", 0.7))
            await self._send(conn, P.msg(P.GEN_RESULT, rid=rid, **res))
        except Exception as exc:
            await self._send(conn, P.msg(P.GEN_RESULT, rid=rid, error=f"relay_link_failure: {exc}"))

    async def _handle_gen_chunk(self, conn: Connection, data: Dict[str, Any]) -> None:
        sink = self._stream_sinks.get(P.request_id_of(data) or "")
        if sink is not None and data.get("text"):
            try:
                sink(data["text"])
            except Exception:
                pass

    async def _handle_gen_terminal(self, conn: Connection, data: Dict[str, Any]) -> None:
        rid = P.request_id_of(data)
        fut = self._pending_requests.get(rid or "")
        if fut is not None and not fut.done():
            fut.set_result({k: v for k, v in data.items() if k not in ("type",)})

    # ------------------------------------------------------------- byte pieces
    async def publish_blob(self, data: bytes, piece_size: int = BLOB_PIECE_SIZE) -> str:
        chunks = split_pieces(data, piece_size)
        h = sha256_hex_bytes(data)
        self.pieces[h] = {"hashes": piece_hashes(chunks), "size": len(data), "chunks": chunks}
        await announce_piece(self.dht, h, self.addr or self.peer_id)
        return h

    async def _handle_piece_request(self, conn: Connection, data: Dict[str, Any]) -> None:
        h, idx = data.get("content_hash"), data.get("index")
        blob = self.pieces.get(h)
        if blob is None:
            await self._send(conn, P.msg(P.PIECE_DATA, content_hash=h, index=idx, error="unknown_content"))
            return
        if idx is None:          # manifest request
            await self._send(conn, P.msg(P.PIECE_DATA, content_hash=h, index=None, hashes=blob["hashes"],
                                         size=blob["size"]))
            return
        if not (0 <= int(idx) < len(blob["chunks"])):
            await self._send(conn, P.msg(P.PIECE_DATA, content_hash=h, index=idx, error="bad_index"))
            return
        payload = base64.b64encode(blob["chunks"][int(idx)]).decode()
        await self._send(conn, P.msg(P.PIECE_DATA, content_hash=h, index=int(idx), data=payload))

    async def _handle_piece_data(self, conn: Connection, data: Dict[str, Any]) -> None:
        st = self._pending_blobs.get(data.get("content_hash") or "")
        if st is None:
            return
        if data.get("error"):
            st["error"] = data["error"]
        elif data.get("index") is None:
            st["hashes"], st["size"] = data.get("hashes") or [], data.get("size", 0)
        else:
            st["chunks"][int(data["index"])] = base64.b64decode(data.get("data") or "")
        st["event"].set()

    async def fetch_blob(self, pid: str, content_hash: str, timeout: float = 30.0) -> bytes:
        """Download a published blob from ``pid`` piece by piece and verify every hash."""
        conn = self._conn_of(pid)
        if conn is None:
            raise ConnectionError(f"not connected to {pid}")
        st: Dict[str, Any] = {"chunks": {}, "event": asyncio.Event(), "hashes": None}
        self._pending_blobs[content_hash] = st
        try:
            await self._send(conn, P.msg(P.PIECE_REQUEST, content_hash=content_hash, index=None))
            await asyncio.wait_for(st["event"].wait(), timeout)
            if st.get("error"):
                raise ServiceError(st["error"])
            for i in range(len(st["hashes"])):
                st["event"].clear()
                await self._send(conn, P.msg(P.PIECE_REQUEST, content_hash=content_hash, index=i))
                while i not in st["chunks"] and not st.get("error"):
                    await asyncio.wait_for(st["event"].wait(), timeout)
                    st["event"].clear()
                if st.get("error"):
                    raise ServiceError(st["error"])
            blob = verify_and_reassemble([st["chunks"][i] for i in range(len(st["hashes"]))], st["hashes"])
            if sha256_hex_bytes(blob) != content_hash:
                raise ValueError("content_hash_mismatch")
            return blob
        finally:
            self._pending_blobs.pop(content_hash, None)

    # ------------------------------------------------ CPU/loopback activation hop
    async def _handle_hidden_forward(self, conn: Connection, data: Dict[str, Any]) -> None:
        from .parallel.cpu_pipeline import decode_tensor, encode_tensor

        host = self.piece_hosts.get(data.get("piece_key") or "")
        rid = data.get("rid")
        if host is None:
            await self._send(conn, P.msg(P.HIDDEN_RESULT, rid=rid, error="unknown_piece"))
            return
        try:
            x = decode_tensor(data["tensor"])
            loop = asyncio.get_running_loop()
            y = await loop.run_in_executor(None, host.forward, data.get("session"), x, data.get("positions"),
                                           bool(data.get("reset")), bool(data.get("release")))
            await self._send(conn, P.msg(P.HIDDEN_RESULT, rid=rid, tensor=encode_tensor(y) if y is not None else None))
        except Exception as exc:
            await self._send(conn, P.msg(P.HIDDEN_RESULT, rid=rid, error=f"piece_error: {exc}"))

    async def _handle_hidden_result(self, conn: Connection, data: Dict[str, Any]) -> None:
        fut = self._pending_hidden.pop(data.get("rid") or "", None)
        if fut is not None and not fut.done():
            fut.set_result(data)

    async def forward_hidden(self, pid: str, piece_key: str, session: str, tensor_payload: Dict[str, Any],
                             positions: List[int], reset: bool = False, release: bool = False,
                             timeout: float = 120.0) -> Dict[str, Any]:
        conn = self._conn_of(pid)
        if conn is None:
            raise ConnectionError(f"not connected to {pid}")
        rid = new_id("hid")
        fut = asyncio.get_running_loop().create_future()
        self._pending_hidden[rid] = fut
        await self._send(conn, P.msg(P.HIDDEN_FORWARD, rid=rid, piece_key=piece_key, session=session,
                                     tensor=tensor_payload, positions=positions, reset=reset, release=release))
        res = await asyncio.wait_for(fut, timeout)
        if res.get("error"):
            raise ServiceError(res["error"])
        return res

    # =============================================================== public API
    def list_providers(self) -> List[Dict[str, Any]]:
        out = []
        for pid, svcs in list(self.providers.items()):
            models: List[str] = []
            price, tag, found = float("inf"), None, False
            for name, meta in svcs.items():
                if name.startswith("_") or not isinstance(meta, dict) or "models" not in meta:
                    continue
                found = True
                models.extend(meta.get("models") or [])
                price = min(price, float(meta.get("price_per_token", 0.0) or 0.0))
                tag = tag or meta.get("tag")
            if found:
                out.append({"peer_id": pid, "addr": self.addr if pid == self.peer_id else (self.peers.get(pid) or {}).get("addr"),
                            "latency_ms": svcs.get("_latency"), "models": sorted(set(models)),
                            "price_per_token": 0.0 if price == float("inf") else price, "tag": tag})
        return out

    def pick_provider(self, model_name: str) -> Optional[Tuple[str, Dict[str, Any]]]:
        """Cheapest, then lowest-latency provider of ``model_name`` (p2p_runtime.py:723-757);
        degraded providers sort last."""
        cands = []
        for pid, svcs in self.providers.items():
            for name, meta in svcs.items():
                if name.startswith("_") or not isinstance(meta, dict):
                    continue
                if model_name in (meta.get("models") or []):
                    lat = svcs.get("_latency")
                    cands.append((svcs.get("health") == "degraded" or meta.get("healthy") is False,
                                  float(meta.get("price_per_token", 0.0) or 0.0),
                                  99999.0 if lat is None else float(lat), pid, name))
                    break
        if not cands:
            return None
        cands.sort(key=lambda c: c[:3])
        _, _, _, pid, name = cands[0]
        meta = dict(self.providers[pid][name])
        meta["_svc_name"] = name
        return pid, meta

    async def request_generation(self, provider_id: str, prompt: str, max_new_tokens: int = 32,
                                 model_name: Optional[str] = None, temperature: float = 0.7, stream: bool = False,
                                 on_chunk: Optional[Callable[[str], None]] = None,
                                 timeout: float = DEFAULT_GEN_TIMEOUT) -> Dict[str, Any]:
        params = {"prompt": prompt, "max_new_tokens": max_new_tokens, "temperature": temperature}
        if provider_id == self.peer_id:
            svc = self._find_local_service(None, model_name)
            if svc is None:
                raise ServiceError(f"no local service for model {model_name}")
            if stream and on_chunk is not None:
                text = []
                async for raw in svc.aexecute_stream(params):
                    try:
                        obj = json.loads(raw)
                        piece = obj.get("text", "") if isinstance(obj, dict) else raw
                    except ValueError:
                        piece = raw
                    if piece:
                        on_chunk(piece)
                        text.append(piece)
                return {"text": "".join(text)}
            return await svc.aexecute(params)
        conn = self._conn_of(provider_id)
        if conn is None:
            raise ConnectionError(f"Provider {provider_id} not connected")
        rid = new_id("req")
        fut = asyncio.get_running_loop().create_future()
        fut._b2b_peer = provider_id                      # type: ignore[attr-defined]
        self._pending_requests[rid] = fut
        if on_chunk is not None:
            self._stream_sinks[rid] = on_chunk
        svc_name = "hf"
        for name, meta in (self.providers.get(provider_id) or {}).items():
            if not name.startswith("_") and isinstance(meta, dict) and (
                    not model_name or model_name in (meta.get("models") or [])):
                svc_name = name
                break
        try:
            ok = await self._send(conn, P.gen_request(rid, prompt, model=model_name, svc=svc_name,
                                                      max_new_tokens=max_new_tokens, temperature=temperature,
                                                      stream=bool(stream or on_chunk)))
            if not ok:
                raise ConnectionError(f"send to {provider_id} failed")
            res = await asyncio.wait_for(fut, timeout)
        finally:
            self._pending_requests.pop(rid, None)
            self._stream_sinks.pop(rid, None)
        if res.get("error"):
            raise ServiceError(str(res["error"]))
        res.pop("rid", None)
        return res

    def mesh_topology(self) -> Dict[str, Any]:
        """peer_id <-> address <-> hosted layer pieces (the NVLink topology table's control-plane view)."""
        table = {self.peer_id: {"addr": self.addr, "pieces": [p.describe() for p in self.layer_pieces]}}
        for pid, info in self.peers.items():
            table[pid] = {"addr": info.get("addr"), "pieces": self.remote_layer_pieces.get(pid, []),
                          "latency_ms": info.get("last_pong_ms")}
        return table

    def uptime(self) -> float:
        return time.time() - self.start_time if self.start_time else 0.0


# ==================================================================================== launcher
async def run_p2p_node(host: str = "0.0.0.0", port: int = 0, bootstrap_link: Optional[str] = None,
                       model_name: Optional[str] = None, price_per_token: float = 0.0, backend: str = "hf",
                       announce_host: Optional[str] = None, announce_port: Optional[int] = None,
                       region: str = "Auto", api_port: Optional[int] = None, api_host: str = "0.0.0.0",
                       token: Optional[str] = None, pieces: int = 1, transport: str = "ws",
                       serve_forever: bool = True, ready: Optional[asyncio.Event] = None,
                       service_kw: Optional[Dict[str, Any]] = None) -> P2PNode:
    """Bring a provider node up (parity: p2p_runtime.py:843-954): mesh listener, optional API
    sidecar in the same loop sharing the node, bootstrap, model load off-loop, announce, join
    link + registration URL, registry sync, heartbeat."""
    node = P2PNode(host=host, port=port, announce_host=announce_host, announce_port=announce_port, region=region,
                   transport=transport)
    node.api_port, node.api_host = api_port, api_host
    await node.start()
    api_task = None
    if api_port:
        import uvicorn

        from . import api as api_mod

        api_mod.node = node
        config = uvicorn.Config(api_mod.app, host=api_host, port=api_port, log_level="warning", lifespan="on")
        server = uvicorn.Server(config)
        api_task = asyncio.create_task(server.serve())
        node._tasks.append(api_task)
        node._api_server = server                         # type: ignore[attr-defined]
    if bootstrap_link:
        await node.connect_bootstrap(bootstrap_link)
    if model_name:
        kw = dict(service_kw or {})
        if backend == "hf":
            kw.setdefault("pieces", pieces)
            kw["price_per_token"] = price_per_token
        if backend == "hf_remote":
            kw["token"] = token
        svc = build_service(backend, model_name, **kw)
        await asyncio.get_running_loop().run_in_executor(None, svc.load_sync)      # keeps pings alive
        await node.add_service(svc)
        link = generate_join_link("connectit", model_name, sha256_hex(model_name), [node.addr])
        node.join_link = link                                                      # type: ignore[attr-defined]
        try:
            from rich.console import Console

            con = Console()
            con.print(f"[bold green]Node ready[/bold green]  peer={node.peer_id}  addr={node.addr}  model={model_name}")
            con.print(f"Join link: {link}")
            con.print(f"Register:  {registration_url(link, region, backend, api_port or 0)}")
        except Exception:
            print(f"Join link: {link}")
    if node.registry.enabled:
        await node.sync_with_registry()
    if ready is not None:
        ready.set()
    if not serve_forever:
        return node
    try:
        while True:
            await asyncio.sleep(15)
            logger.debug(f"heartbeat peers={len(node.peers)} providers={len(node.providers)}")
    finally:
        await node.stop()
    return node


def main(argv: Optional[List[str]] = None) -> None:
    """``python -m bee2bee_b200.p2p_runtime --register --model M --provider hf|ollama ...``
    (parity: p2p_runtime.py:956-980, used by run.sh)."""
    import argparse

    ap = argparse.ArgumentParser()
    ap.add_argument("--register", action="store_true")
    ap.add_argument("--model", default="distilgpt2")
    ap.add_argument("--provider", default="hf", choices=["hf", "ollama", "hf_remote"])
    ap.add_argument("--endpoint", default=None, help="Ollama host, e.g. http://localhost:11434")
    ap.add_argument("--tag", default="global")
    ap.add_argument("--port", type=int, default=0)
    ap.add_argument("--api-port", type=int, default=None)
    ap.add_argument("--bootstrap", default=None)
    ap.add_argument("--pieces", type=int, default=1)
    a = ap.parse_args(argv)
    if a.endpoint and a.provider == "ollama":
        os.environ["OLLAMA_HOST"] = a.endpoint
    asyncio.run(run_p2p_node(port=a.port, bootstrap_link=a.bootstrap, model_name=a.model, backend=a.provider,
                             api_port=a.api_port, pieces=a.pieces))


if __name__ == "__main__":
    main()
