"""ROS1 bag (format 2.0) reader/writer in plain Python, for feeding recorded runs to the replay loop.

The reference node takes its inputs from two topics and can record its outputs
(``ratslam/ros_simulate.py:82-83`` subscribers, ``:92-95,116-117,132,147-149`` ``rosbag.Bag.write``):

=========================  ====================  =======================================================
topic                      type                  used as
=========================  ====================  =======================================================
``navbot/camera/image``    sensor_msgs/Image     ``bridge.imgmsg_to_cv(data, "mono8")`` (:100-101)
``navbot/odom``            nav_msgs/Odometry     ``data.twist.twist`` -> (linear.x, angular.z) (:126-129)
``navbot/templatematches`` std_msgs/Int32        index of the matched / created template (:111-113)
``navbot/experiencemap``   geometry_msgs/Pose2D  current experience-map point (:142-143)
=========================  ====================  =======================================================

``rosbag``/``rospy``/``cv_bridge`` are not available (and are transport, not the hot path), so this module
restates the published container format -- ``#ROSBAG V2.0``, records of ``<header_len><header><data_len><data>``
with ``name=value`` header fields, op codes 0x02 message, 0x03 bag header, 0x04 index, 0x05 chunk (``none`` or
``bz2``), 0x06 chunk info, 0x07 connection -- and the ROS1 wire serialisation of the four message types above.
Nothing here touches the GPU; frames leave as uint8 arrays and are sub-sampled on the device
(``prs_vt_extract_u8``).
"""
from __future__ import annotations

import bz2
import struct
from collections import namedtuple

import numpy as np

MAGIC = b"#ROSBAG V2.0\n"
OP_MSG, OP_BAG_HEADER, OP_INDEX, OP_CHUNK, OP_CHUNK_INFO, OP_CONNECTION = 0x02, 0x03, 0x04, 0x05, 0x06, 0x07

IMAGE_TOPIC = "navbot/camera/image"
ODOM_TOPIC = "navbot/odom"
MATCH_TOPIC = "navbot/templatematches"
EM_TOPIC = "navbot/experiencemap"

# type name -> (md5sum, message definition text) as the ROS message generators publish them
MSG_TYPES = {
    "sensor_msgs/Image": ("060021388200f6f0f447d0fcd9c64743",
                          "Header header\nuint32 height\nuint32 width\nstring encoding\nuint8 is_bigendian\n"
                          "uint32 step\nuint8[] data\n"),
    "nav_msgs/Odometry": ("cd5e73d190d741a2f92e81eda573aca7",
                          "Header header\nstring child_frame_id\ngeometry_msgs/PoseWithCovariance pose\n"
                          "geometry_msgs/TwistWithCovariance twist\n"),
    "std_msgs/Int32": ("da5909fbe378aeaf85e547e830cc1bb7", "int32 data\n"),
    "geometry_msgs/Pose2D": ("938fa65709584ad8e77d238529be13b8", "float64 x\nfloat64 y\nfloat64 theta\n"),
}

Message = namedtuple("Message", "topic msgtype stamp data")      # stamp = (secs, nsecs) of the bag record
Image = namedtuple("Image", "stamp frame_id encoding image")     # image: uint8 [H, W] (mono8)
Odometry = namedtuple("Odometry", "stamp frame_id child_frame_id position orientation linear angular")


class BagFormatError(ValueError):
    pass


# ---------------------------------------------------------------------------------------------- records
def _pack_header(fields):
    out = bytearray()
    for name, value in fields.items():
        item = name.encode("ascii") + b"=" + value
        out += struct.pack("<I", len(item)) + item
    return bytes(out)


def _parse_header(buf):
    fields, pos = {}, 0
    while pos < len(buf):
        if pos + 4 > len(buf):
            raise BagFormatError("truncated header field length")
        (n,) = struct.unpack_from("<I", buf, pos)
        pos += 4
        item = buf[pos:pos + n]
        if len(item) != n or b"=" not in item:
            raise BagFormatError("malformed header field")
        pos += n
        name, value = item.split(b"=", 1)
        fields[name.decode("ascii")] = bytes(value)
    return fields


def _record(fields, data):
    h = _pack_header(fields)
    return struct.pack("<I", len(h)) + h + struct.pack("<I", len(data)) + data


def _records(buf, pos=0, end=None):
    """Yield (header fields, data bytes, offset) for the records laid end to end in ``buf[pos:end]``."""
    end = len(buf) if end is None else end
    while pos < end:
        start = pos
        if pos + 4 > end:
            raise BagFormatError("truncated record at offset %d" % pos)
        (hl,) = struct.unpack_from("<I", buf, pos)
        pos += 4
        if pos + hl + 4 > end:
            raise BagFormatError("truncated record header at offset %d" % start)
        fields = _parse_header(buf[pos:pos + hl])
        pos += hl
        (dl,) = struct.unpack_from("<I", buf, pos)
        pos += 4
        if pos + dl > end:
            raise BagFormatError("truncated record data at offset %d" % start)
        yield fields, buf[pos:pos + dl], start
        pos += dl


def _u32(b):
    return struct.unpack("<I", b)[0]


def _time(b):
    return struct.unpack("<II", b)


# ---------------------------------------------------------------------------------------------- reader
class BagReader(object):
    """Sequential reader: every chunk is decompressed and scanned once; the index records are not needed."""

    def __init__(self, path):
        with open(path, "rb") as f:
            self._buf = f.read()
        if not self._buf.startswith(MAGIC):
            raise BagFormatError("not a ROS bag v2.0 file: %r" % (path,))
        self.connections = {}           # conn id -> dict(topic=..., type=..., md5sum=...)
        self.chunk_count = 0
        self._messages = []
        self._scan()

    def _connection(self, fields, data):
        info = _parse_header(data)
        self.connections[_u32(fields["conn"])] = {
            "topic": fields["topic"].decode(), "type": info.get("type", b"").decode(),
            "md5sum": info.get("md5sum", b"").decode()}

    def _scan(self):
        order = 0
        for fields, data, _ in _records(self._buf, len(MAGIC)):
            op = fields["op"][0]
            if op == OP_CHUNK:
                comp = fields["compression"].decode()
                if comp == "bz2":
                    data = bz2.decompress(data)
                elif comp != "none":
                    raise BagFormatError("chunk compression %r is not supported (none, bz2)" % comp)
                if len(data) != _u32(fields["size"]):
                    raise BagFormatError("chunk size field does not match its data")
                self.chunk_count += 1
                for f2, d2, _ in _records(data):
                    op2 = f2["op"][0]
                    if op2 == OP_CONNECTION:
                        self._connection(f2, d2)
                    elif op2 == OP_MSG:
                        self._messages.append((_time(f2["time"]), order, _u32(f2["conn"]), d2))
                        order += 1
            elif op == OP_CONNECTION:
                self._connection(fields, data)
            elif op == OP_MSG:            # unchunked message (not written by rosbag >= 1.1, accepted anyway)
                self._messages.append((_time(fields["time"]), order, _u32(fields["conn"]), data))
                order += 1
        self._messages.sort(key=lambda m: (m[0], m[1]))     # bag time, ties in file order

    @property
    def topics(self):
        return sorted({c["topic"] for c in self.connections.values()})

    def __len__(self):
        return len(self._messages)

    def messages(self, topics=None):
        """Yield ``Message`` tuples in bag-time order (``rosbag.Bag.read_messages`` order)."""
        want = None if topics is None else set(topics)
        for stamp, _, conn, data in self._messages:
            c = self.connections.get(conn)
            if c is None:
                raise BagFormatError("message on unknown connection %d" % conn)
            if want is None or c["topic"] in want:
                yield Message(c["topic"], c["type"], stamp, data)


# ---------------------------------------------------------------------------------------------- writer
class BagWriter(object):
    """Writes chunked bags (``none`` or ``bz2``) with index and chunk-info records, like ``rosbag.Bag(path, 'w')``."""

    def __init__(self, path, compression="none", chunk_threshold=768 * 1024):
        if compression not in ("none", "bz2"):
            raise ValueError("compression must be 'none' or 'bz2'")
        self._f = open(path, "wb")
        self._compression = compression
        self._threshold = chunk_threshold
        self._conns = {}                 # (topic, type) -> id
        self._conn_records = []
        self._chunk = bytearray()
        self._chunk_conns = set()
        self._chunk_index = {}           # conn -> [(stamp, offset)]
        self._chunk_infos = []
        self._f.write(MAGIC)
        self._f.write(self._bag_header(0, 0, 0))

    @staticmethod
    def _bag_header(index_pos, conn_count, chunk_count):
        h = _pack_header({"op": bytes([OP_BAG_HEADER]), "index_pos": struct.pack("<Q", index_pos),
                          "conn_count": struct.pack("<I", conn_count), "chunk_count": struct.pack("<I", chunk_count)})
        pad = 4096 - 4 - len(h) - 4      # the bag header record always occupies 4096 bytes
        return struct.pack("<I", len(h)) + h + struct.pack("<I", pad) + b" " * pad

    def _conn_record(self, cid, topic, msgtype):
        md5, definition = MSG_TYPES.get(msgtype, ("*", ""))
        data = _pack_header({"topic": topic.encode(), "type": msgtype.encode(), "md5sum": md5.encode(),
                             "message_definition": definition.encode()})
        return _record({"op": bytes([OP_CONNECTION]), "conn": struct.pack("<I", cid), "topic": topic.encode()}, data)

    def write(self, topic, msgtype, stamp, data):
        """Append one serialised message; ``stamp`` = (secs, nsecs)."""
        key = (topic, msgtype)
        cid = self._conns.get(key)
        if cid is None:
            cid = self._conns[key] = len(self._conns)
            self._conn_records.append(self._conn_record(cid, topic, msgtype))
        if cid not in self._chunk_conns:  # a chunk carries the connection record of every connection it uses
            self._chunk_conns.add(cid)
            self._chunk += self._conn_records[cid]
        self._chunk_index.setdefault(cid, []).append((stamp, len(self._chunk)))
        self._chunk += _record({"op": bytes([OP_MSG]), "conn": struct.pack("<I", cid),
                                "time": struct.pack("<II", *stamp)}, bytes(data))
        if len(self._chunk) >= self._threshold:
            self._flush()

    def _flush(self):
        if not self._chunk_index:
            return
        raw = bytes(self._chunk)
        payload = bz2.compress(raw) if self._compression == "bz2" else raw
        pos = self._f.tell()
        self._f.write(_record({"op": bytes([OP_CHUNK]), "compression": self._compression.encode(),
                               "size": struct.pack("<I", len(raw))}, payload))
        stamps = [s for entries in self._chunk_index.values() for s, _ in entries]
        counts = b""
        for cid, entries in sorted(self._chunk_index.items()):
            body = b"".join(struct.pack("<III", s[0], s[1], off) for s, off in entries)
            self._f.write(_record({"op": bytes([OP_INDEX]), "ver": struct.pack("<I", 1), "conn": struct.pack("<I", cid),
                                   "count": struct.pack("<I", len(entries))}, body))
            counts += struct.pack("<II", cid, len(entries))
        self._chunk_infos.append(_record(
            {"op": bytes([OP_CHUNK_INFO]), "ver": struct.pack("<I", 1), "chunk_pos": struct.pack("<Q", pos),
             "start_time": struct.pack("<II", *min(stamps)), "end_time": struct.pack("<II", *max(stamps)),
             "count": struct.pack("<I", len(self._chunk_index))}, counts))
        self._chunk = bytearray()
        self._chunk_conns = set()
        self._chunk_index = {}

    def close(self):
        if self._f is None:
            return
        self._flush()
        index_pos = self._f.tell()
        for r in self._conn_records:
            self._f.write(r)
        for r in self._chunk_infos:
            self._f.write(r)
        self._f.seek(len(MAGIC))
        self._f.write(self._bag_header(index_pos, len(self._conn_records), len(self._chunk_infos)))
        self._f.close()
        self._f = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


# ---------------------------------------------------------------------------------------------- messages
class _Cursor(object):
    def __init__(self, buf):
        self.buf, self.pos = buf, 0

    def take(self, fmt):
        vals = struct.unpack_from(fmt, self.buf, self.pos)
        self.pos += struct.calcsize(fmt)
        return vals

    def string(self):
        (n,) = self.take("<I")
        s = self.buf[self.pos:self.pos + n]
        if len(s) != n:
            raise BagFormatError("truncated string/array in message")
        self.pos += n
        return s


def _ser_header(seq, stamp, frame_id):
    fid = frame_id.encode()
    return struct.pack("<III", seq, stamp[0], stamp[1]) + struct.pack("<I", len(fid)) + fid


def _to_mono8(raw, height, width, step, encoding, big_endian):
    """What ``CvBridge.imgmsg_to_cv(msg, "mono8")`` hands the node: cvtColor's fixed-point luma for colour
    encodings (Y = (R*4899 + G*9617 + B*1868 + 8192) >> 14), 255/65535 scaling for 16-bit grey."""
    enc = encoding.lower()
    chan = {"mono8": 1, "8uc1": 1, "rgb8": 3, "bgr8": 3, "rgba8": 4, "bgra8": 4, "mono16": 2, "16uc1": 2}.get(enc)
    if chan is None:
        raise BagFormatError("image encoding %r is not supported" % encoding)
    if step < width * chan or len(raw) < step * height:
        raise BagFormatError("image data shorter than height*step")
    rows = np.frombuffer(raw, np.uint8, step * height).reshape(height, step)[:, :width * chan]
    if enc in ("mono8", "8uc1"):
        return np.ascontiguousarray(rows)
    if enc in ("mono16", "16uc1"):
        v = rows.reshape(height, width, 2).astype(np.uint32)
        v16 = (v[..., 0] << 8 | v[..., 1]) if big_endian else (v[..., 1] << 8 | v[..., 0])
        return np.clip(np.rint(v16 * (255.0 / 65535.0)), 0, 255).astype(np.uint8)
    px = rows.reshape(height, width, chan).astype(np.uint32)
    r, g, b = (px[..., 0], px[..., 1], px[..., 2]) if enc.startswith("rgb") else (px[..., 2], px[..., 1], px[..., 0])
    return ((r * 4899 + g * 9617 + b * 1868 + 8192) >> 14).astype(np.uint8)


def decode_image(data):
    c = _Cursor(data)
    _, secs, nsecs = c.take("<III")
    frame_id = c.string().decode(errors="replace")
    height, width = c.take("<II")
    encoding = c.string().decode()
    (big_endian,) = c.take("<B")
    (step,) = c.take("<I")
    raw = c.string()
    return Image((secs, nsecs), frame_id, encoding, _to_mono8(raw, height, width, step, encoding, bool(big_endian)))


def encode_image(image, stamp=(0, 0), seq=0, frame_id="camera", encoding="mono8"):
    a = np.ascontiguousarray(image)
    if encoding == "mono8":
        if a.dtype != np.uint8 or a.ndim != 2:
            raise ValueError("mono8 needs a uint8 [H, W] array")
        step = a.shape[1]
    elif encoding in ("rgb8", "bgr8"):
        if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3:
            raise ValueError("%s needs a uint8 [H, W, 3] array" % encoding)
        step = a.shape[1] * 3
    elif encoding == "mono16":
        if a.dtype != np.uint16 or a.ndim != 2:
            raise ValueError("mono16 needs a uint16 [H, W] array")
        a = a.astype("<u2")
        step = a.shape[1] * 2
    else:
        raise ValueError("unsupported encoding %r" % encoding)
    enc = encoding.encode()
    raw = a.tobytes()
    return (_ser_header(seq, stamp, frame_id) + struct.pack("<II", a.shape[0], a.shape[1]) +
            struct.pack("<I", len(enc)) + enc + struct.pack("<BI", 0, step) + struct.pack("<I", len(raw)) + raw)


def decode_odometry(data):
    c = _Cursor(data)
    _, secs, nsecs = c.take("<III")
    frame_id = c.string().decode(errors="replace")
    child = c.string().decode(errors="replace")
    position = c.take("<3d")
    orientation = c.take("<4d")
    c.take("<36d")
    linear = c.take("<3d")
    angular = c.take("<3d")
    c.take("<36d")
    return Odometry((secs, nsecs), frame_id, child, position, orientation, linear, angular)


def encode_odometry(linear_x, angular_z, stamp=(0, 0), seq=0, frame_id="odom", child_frame_id="base_link",
                    position=(0.0, 0.0, 0.0), orientation=(0.0, 0.0, 0.0, 1.0)):
    child = child_frame_id.encode()
    cov = struct.pack("<36d", *([0.0] * 36))
    return (_ser_header(seq, stamp, frame_id) + struct.pack("<I", len(child)) + child +
            struct.pack("<3d", *position) + struct.pack("<4d", *orientation) + cov +
            struct.pack("<3d", float(linear_x), 0.0, 0.0) + struct.pack("<3d", 0.0, 0.0, float(angular_z)) + cov)


def encode_int32(value):
    return struct.pack("<i", int(value))


def decode_int32(data):
    return struct.unpack_from("<i", data)[0]


def encode_pose2d(x, y, theta=0.0):
    return struct.pack("<3d", float(x), float(y), float(theta))


def decode_pose2d(data):
    return struct.unpack_from("<3d", data)


# ---------------------------------------------------------------------------------------------- front end
def read_events(path, image_topic=IMAGE_TOPIC, odom_topic=ODOM_TOPIC):
    """The node's input messages in bag-time order: ``("odom", stamp, (linear.x, angular.z))`` and
    ``("image", stamp, uint8[H, W])``.  A leading ``/`` in topic names is ignored."""
    bag = BagReader(path)
    want = {image_topic.lstrip("/"): "image", odom_topic.lstrip("/"): "odom"}
    events = []
    for m in bag.messages():
        kind = want.get(m.topic.lstrip("/"))
        if kind == "image":
            events.append(("image", m.stamp, decode_image(m.data).image))
        elif kind == "odom":
            o = decode_odometry(m.data)
            events.append(("odom", m.stamp, (o.linear[0], o.angular[2])))
    return events


def events_to_arrays(events):
    """``frames[T, H, W]`` uint8, ``odom[T, 2]`` float64, ``stamps[T]`` seconds -- the ``.npy`` form of a run
    (SURVEY config 2).  Frame t is paired with the most recent twist that arrived after frame t-1 (zeros when
    none did, which the node's 0.001 gate then drops); twists that are overwritten before a frame arrives are
    lost, so this is exact only for recordings in which the two topics alternate -- ``replay_events`` keeps
    every message."""
    frames, odom, stamps = [], [], []
    last = (0.0, 0.0)
    for kind, stamp, payload in events:
        if kind == "odom":
            last = payload
        else:
            frames.append(payload)
            odom.append(last)
            stamps.append(stamp[0] + stamp[1] * 1e-9)
            last = (0.0, 0.0)
    if not frames:
        return np.zeros((0, 0, 0), np.uint8), np.zeros((0, 2)), np.zeros(0)
    return np.stack(frames), np.asarray(odom, dtype=np.float64).reshape(-1, 2), np.asarray(stamps)


def iter_frames(path, chunk, image_topic=IMAGE_TOPIC, odom_topic=ODOM_TOPIC):
    """``events_to_arrays(read_events(path, ...))[:2]`` in pieces: yields ``(frames[n, H, W] uint8, odom[n, 2])`` with
    n <= ``chunk`` (n < chunk only for the last piece), paired by the same rule.  Images are decoded only for the piece
    being yielded, so the decoded frames in memory stay at one piece; ``BagReader`` still reads the file whole."""
    chunk = int(chunk)
    if chunk < 1:
        raise ValueError("iter_frames: chunk must be >= 1, got %r" % (chunk,))
    bag = BagReader(path)
    want = {image_topic.lstrip("/"): "image", odom_topic.lstrip("/"): "odom"}
    raw, odom = [], []
    last = (0.0, 0.0)
    for m in bag.messages():
        kind = want.get(m.topic.lstrip("/"))
        if kind == "odom":
            o = decode_odometry(m.data)
            last = (o.linear[0], o.angular[2])
        elif kind == "image":
            raw.append(m.data)
            odom.append(last)
            last = (0.0, 0.0)
            if len(raw) == chunk:
                yield np.stack([decode_image(d).image for d in raw]), np.asarray(odom, dtype=np.float64)
                raw, odom = [], []
    if raw:
        yield np.stack([decode_image(d).image for d in raw]), np.asarray(odom, dtype=np.float64).reshape(-1, 2)


def write_run(path, frames, odom, rate_hz=10.0, compression="none", image_topic=IMAGE_TOPIC, odom_topic=ODOM_TOPIC,
              chunk_threshold=768 * 1024):
    """Write ``frames[T,H,W]`` / ``odom[T,2]`` as the bag the node would have been fed: per time step one
    nav_msgs/Odometry followed by one sensor_msgs/Image."""
    with BagWriter(path, compression=compression, chunk_threshold=chunk_threshold) as w:
        for t in range(len(frames)):
            ns = int(round(t * 1e9 / rate_hz))
            s_odom = (ns // 10 ** 9, ns % 10 ** 9)
            s_img = ((ns + 1000) // 10 ** 9, (ns + 1000) % 10 ** 9)
            w.write(odom_topic, "nav_msgs/Odometry", s_odom,
                    encode_odometry(odom[t][0], odom[t][1], stamp=s_odom, seq=t))
            w.write(image_topic, "sensor_msgs/Image", s_img, encode_image(frames[t], stamp=s_img, seq=t))


def iter_events(path, chunk, image_topic=IMAGE_TOPIC, odom_topic=ODOM_TOPIC):
    """``read_events(path, ...)`` in pieces: yields lists of events holding at most ``chunk`` images each.  A piece ends
    right after its ``chunk``-th image, wherever that falls (the odometry after it opens the next piece), and the last
    piece holds what remains, trailing odometry included; concatenated, the pieces are ``read_events``.  Images are
    decoded only for the piece being yielded; ``BagReader`` still reads the file whole."""
    chunk = int(chunk)
    if chunk < 1:
        raise ValueError("iter_events: chunk must be >= 1, got %r" % (chunk,))
    bag = BagReader(path)
    want = {image_topic.lstrip("/"): "image", odom_topic.lstrip("/"): "odom"}
    piece, n_img = [], 0
    for m in bag.messages():
        kind = want.get(m.topic.lstrip("/"))
        if kind == "odom":
            o = decode_odometry(m.data)
            piece.append(("odom", m.stamp, (o.linear[0], o.angular[2])))
        elif kind == "image":
            piece.append(("image", m.stamp, m.data))
            n_img += 1
            if n_img == chunk:
                yield [(k, s, decode_image(p).image if k == "image" else p) for k, s, p in piece]
                piece, n_img = [], 0
    if piece:
        yield [(k, s, decode_image(p).image if k == "image" else p) for k, s, p in piece]


def write_events(path, events, compression="none", image_topic=IMAGE_TOPIC, odom_topic=ODOM_TOPIC,
                 chunk_threshold=768 * 1024):
    """Write a message stream as ``read_events`` returns it -- ``("odom", stamp, (linear.x, angular.z))`` and
    ``("image", stamp, uint8[H, W])`` -- as a bag, each message at its own stamp, so that ``read_events`` gives the
    stream back."""
    with BagWriter(path, compression=compression, chunk_threshold=chunk_threshold) as w:
        n_odom = n_img = 0
        for kind, stamp, payload in events:
            stamp = (int(stamp[0]), int(stamp[1]))
            if kind == "odom":
                w.write(odom_topic, "nav_msgs/Odometry", stamp,
                        encode_odometry(payload[0], payload[1], stamp=stamp, seq=n_odom))
                n_odom += 1
            elif kind == "image":
                w.write(image_topic, "sensor_msgs/Image", stamp, encode_image(payload, stamp=stamp, seq=n_img))
                n_img += 1
            else:
                raise ValueError("write_events: unknown event kind %r" % (kind,))
