"""Host-side readers for the on-disk formats of the OCT datasets the reference catalogues
(reference ``Datasets.md:3-26``; SURVEY.md 8f-4).  The reference ships no loader code, so these follow
the published file formats, not reference lines:

* MetaImage ``.mhd`` + ``.raw`` / ``.zraw`` (RETOUCH volumes and reference masks): ``read_mhd`` / ``write_mhd``;
* MATLAB ``.mat`` with boundary annotations (Duke DME / AMD: ``manualLayers1`` of shape boundaries x columns x
  B-scans, NaN where a column is not annotated): ``read_mat_layers``;
* Heidelberg Spectralis raw export ``.vol`` (HC-MS, reference ``Datasets.md:13``; also AROI-style Spectralis data):
  ``read_heidelberg_vol`` -- B-scan stack plus the device's own boundary lines;
* HC-MS manual delineations (``.mat`` with ``bd_pts``: columns x B-scans x 9 boundaries): ``read_hcms_delineation``;
* ``.npy`` / ``.npz`` label volumes: ``read_labels``.

Everything here is plain host I/O (numpy, scipy.io for ``.mat``); the arrays go to the GPU through
``suite.evaluate_host`` (label volumes) or ``suite.labels_from_boundaries`` (boundary curves -> label maps).
"""
from __future__ import annotations

import os
import zlib

import numpy as np

_MHD_TYPES = {"MET_UCHAR": np.uint8, "MET_CHAR": np.int8, "MET_USHORT": np.uint16, "MET_SHORT": np.int16,
              "MET_UINT": np.uint32, "MET_INT": np.int32, "MET_FLOAT": np.float32, "MET_DOUBLE": np.float64}
_MHD_NAMES = {np.dtype(v): k for k, v in _MHD_TYPES.items()}


def read_mhd(path):
    """MetaImage header + raw data -> (array in C order ``[..., dim1, dim0]`` = ``[slices, rows, cols]`` for a
    volume, header dict).  Supports ``ElementDataFile = <file> | LOCAL``, ``CompressedData`` (zlib),
    ``BinaryDataByteOrderMSB`` and ``HeaderSize``."""
    with open(path, "rb") as f:
        blob = f.read()
    header, pos = {}, 0
    while True:
        end = blob.find(b"\n", pos)
        if end < 0:
            raise ValueError(f"{path}: no ElementDataFile line")
        line = blob[pos:end].decode("latin-1").strip()
        pos = end + 1
        if not line:
            continue
        if "=" not in line:
            raise ValueError(f"{path}: malformed header line {line!r}")
        key, val = (s.strip() for s in line.split("=", 1))
        header[key] = val
        if key == "ElementDataFile":
            break
    if header.get("ObjectType", "Image") != "Image":
        raise ValueError(f"{path}: ObjectType {header['ObjectType']!r} is not an image")
    ndims = int(header["NDims"])
    dims = [int(v) for v in header["DimSize"].split()]
    if len(dims) != ndims:
        raise ValueError(f"{path}: DimSize has {len(dims)} entries, NDims = {ndims}")
    if header["ElementType"] not in _MHD_TYPES:
        raise ValueError(f"{path}: unsupported ElementType {header['ElementType']}")
    channels = int(header.get("ElementNumberOfChannels", "1"))
    dtype = np.dtype(_MHD_TYPES[header["ElementType"]])
    if header.get("BinaryDataByteOrderMSB", header.get("ElementByteOrderMSB", "False")).lower() == "true":
        dtype = dtype.newbyteorder(">")
    data_file = header["ElementDataFile"]
    if data_file == "LOCAL":
        raw = blob[pos:]
    else:
        if "%" in data_file or data_file == "LIST":
            raise ValueError(f"{path}: one-file-per-slice data ({data_file}) is not supported")
        with open(os.path.join(os.path.dirname(os.path.abspath(path)), data_file), "rb") as f:
            raw = f.read()
    skip = int(header.get("HeaderSize", "0"))
    if skip > 0:
        raw = raw[skip:]
    if header.get("CompressedData", "False").lower() == "true":
        raw = zlib.decompress(raw)
    count = int(np.prod(dims)) * channels
    if len(raw) < count * dtype.itemsize:
        raise ValueError(f"{path}: data file holds {len(raw)} bytes, header needs {count * dtype.itemsize}")
    arr = np.frombuffer(raw, dtype=dtype, count=count)
    shape = tuple(reversed(dims)) + ((channels,) if channels > 1 else ())
    return arr.reshape(shape).astype(dtype.newbyteorder("="), copy=False), header


def mhd_spacing(header):
    """Voxel spacing of a ``read_mhd`` header in the order of the array's axes (``[slices, rows, cols]`` for a volume),
    ready for ``suite.surface_distance_3d(spacing=...)``: the header lists ``ElementSpacing`` fastest axis first (x, y,
    z), so the order is reversed.  KeyError without ``ElementSpacing``, ValueError when it does not have ``NDims``
    numbers."""
    if "ElementSpacing" not in header:
        raise KeyError("the MetaImage header has no ElementSpacing")
    try:
        sp = [float(v) for v in header["ElementSpacing"].split()]
    except ValueError:
        raise ValueError(f"ElementSpacing {header['ElementSpacing']!r} is not a list of numbers") from None
    ndims = int(header.get("NDims", len(sp)))
    if len(sp) != ndims:
        raise ValueError(f"ElementSpacing has {len(sp)} entries, NDims = {ndims}")
    return tuple(reversed(sp))


def write_mhd(path, array, spacing=None, compressed=False):
    """Write ``array`` (C order ``[slices, rows, cols]``) as ``path`` (.mhd) + a sibling .raw / .zraw file."""
    array = np.ascontiguousarray(array)
    if array.dtype not in _MHD_NAMES:
        raise TypeError(f"unsupported dtype {array.dtype}")
    base = os.path.splitext(os.path.basename(path))[0] + (".zraw" if compressed else ".raw")
    payload = array.tobytes()
    if compressed:
        payload = zlib.compress(payload)
    lines = ["ObjectType = Image", f"NDims = {array.ndim}", "BinaryData = True", "BinaryDataByteOrderMSB = False",
             f"CompressedData = {'True' if compressed else 'False'}"]
    if compressed:
        lines.append(f"CompressedDataSize = {len(payload)}")
    if spacing is not None:
        lines.append("ElementSpacing = " + " ".join(str(float(s)) for s in spacing))
    lines += ["DimSize = " + " ".join(str(d) for d in reversed(array.shape)),
              f"ElementType = {_MHD_NAMES[array.dtype]}", f"ElementDataFile = {base}"]
    with open(path, "w", encoding="latin-1", newline="\n") as f:
        f.write("\n".join(lines) + "\n")
    with open(os.path.join(os.path.dirname(os.path.abspath(path)), base), "wb") as f:
        f.write(payload)


def read_mat_layers(path, key=None):
    """Boundary annotations of a Duke-style ``.mat`` file -> float32 ``[B-scans, boundaries, columns]`` with NaN
    where a column is not annotated (ready for ``suite.labels_from_boundaries``), plus the image stack
    ``[B-scans, rows, columns]`` when the file has one (``images``), else None.  ``key`` defaults to the first
    of ``manualLayers1``, ``manualLayers2``, ``automaticLayersDME``, ``automaticLayersNormal``, ``layerMaps``."""
    from scipy.io import loadmat            # scipy is a dependency of the reference's own stack
    mat = loadmat(path)
    names = [key] if key else ["manualLayers1", "manualLayers2", "automaticLayersDME", "automaticLayersNormal", "layerMaps"]
    found = next((n for n in names if n in mat), None)
    if found is None:
        raise KeyError(f"{path}: none of {names} present (variables: {sorted(k for k in mat if not k.startswith('__'))})")
    layers = np.asarray(mat[found], dtype=np.float32)
    if layers.ndim != 3:
        raise ValueError(f"{path}: {found} has shape {layers.shape}, expected 3 dimensions")
    if found == "layerMaps":                 # AMD set: B-scans x columns x boundaries
        layers = np.transpose(layers, (0, 2, 1))
    else:                                    # DME set: boundaries x columns x B-scans
        layers = np.transpose(layers, (2, 0, 1))
    images = None
    if "images" in mat and np.asarray(mat["images"]).ndim == 3:
        images = np.transpose(np.asarray(mat["images"]), (2, 0, 1))     # rows x columns x B-scans on disk
    return np.ascontiguousarray(layers), images


_VOL_HEADER = 2048          # bytes; little-endian throughout
_VOL_INVALID = 3.0e38       # Heidelberg marks missing samples / boundary points with FLT_MAX


def read_heidelberg_vol(path):
    """Heidelberg Engineering raw export (``.vol``, "HSF-OCT-1xx") -> dict with

    * ``bscans``      float32 ``[NumBScans, SizeZ, SizeX]`` (rows = depth samples, invalid samples NaN),
    * ``boundaries``  float32 ``[NumBScans, NumSeg, SizeX]`` -- the device's own boundary lines in pixels (ILM, BM, ...;
      NaN where the device found none), ready for ``suite.labels_from_boundaries`` / ``suite.boundary_metrics``,
    * ``scale``       (ScaleX, Distance between B-scans, ScaleZ) in mm, and ``header`` with the raw fields read.

    Layout (file header 2048 B, then the SLO image, then per B-scan a header of ``BScanHdrSize`` bytes followed by
    ``SizeX * SizeZ`` float32 samples): version 12s @0, SizeX i @12, NumBScans i @16, SizeZ i @20, ScaleX d @24,
    Distance d @32, ScaleZ d @40, SizeXSlo i @48, SizeYSlo i @52, ..., BScanHdrSize i @100; B-scan header: version
    12s @0, BScanHdrSize i @12, StartX/StartY/EndX/EndY d @16..47, NumSeg i @48, OffSeg i @52, Quality f @56, boundary
    lines = NumSeg x SizeX float32 at OffSeg.  Written from the published description of the format; no Spectralis file
    is available offline, the reader is exercised on files synthesised by the tests with the same layout."""
    import struct
    with open(path, "rb") as f:
        blob = f.read()
    if len(blob) < _VOL_HEADER or not blob[:7] == b"HSF-OCT":
        raise ValueError(f"{path}: not a Heidelberg .vol file (version field {blob[:12]!r})")
    size_x, n_scans, size_z = struct.unpack_from("<iii", blob, 12)
    scale_x, distance, scale_z = struct.unpack_from("<ddd", blob, 24)
    slo_x, slo_y = struct.unpack_from("<ii", blob, 48)
    (hdr_size,) = struct.unpack_from("<i", blob, 100)
    if min(size_x, n_scans, size_z) < 1 or hdr_size < 64 or slo_x < 0 or slo_y < 0:
        raise ValueError(f"{path}: implausible header (SizeX {size_x}, NumBScans {n_scans}, SizeZ {size_z}, BScanHdrSize {hdr_size})")
    pos = _VOL_HEADER + slo_x * slo_y
    per_scan = hdr_size + size_x * size_z * 4
    if len(blob) < pos + n_scans * per_scan:
        raise ValueError(f"{path}: file holds {len(blob)} bytes, header needs {pos + n_scans * per_scan}")
    bscans = np.empty((n_scans, size_z, size_x), np.float32)
    lines, n_seg_max = [], 0
    for i in range(n_scans):
        base = pos + i * per_scan
        n_seg, off_seg = struct.unpack_from("<ii", blob, base + 48)
        if n_seg < 0 or n_seg > 32 or off_seg < 0 or off_seg + n_seg * size_x * 4 > hdr_size:
            raise ValueError(f"{path}: B-scan {i}: implausible NumSeg {n_seg} / OffSeg {off_seg}")
        seg = np.frombuffer(blob, "<f4", n_seg * size_x, base + off_seg).reshape(n_seg, size_x).copy()
        seg[seg > _VOL_INVALID] = np.nan
        lines.append(seg)
        n_seg_max = max(n_seg_max, n_seg)
        img = np.frombuffer(blob, "<f4", size_x * size_z, base + hdr_size).reshape(size_z, size_x)
        bscans[i] = np.where(img > _VOL_INVALID, np.nan, img)
    boundaries = np.full((n_scans, n_seg_max, size_x), np.nan, np.float32)
    for i, seg in enumerate(lines):
        boundaries[i, :len(seg)] = seg
    header = {"version": blob[:12].rstrip(b"\0").decode("latin-1"), "SizeX": size_x, "NumBScans": n_scans, "SizeZ": size_z,
              "SizeXSlo": slo_x, "SizeYSlo": slo_y, "BScanHdrSize": hdr_size}
    return {"bscans": bscans, "boundaries": boundaries, "scale": (scale_x, distance, scale_z), "header": header}


def read_hcms_delineation(path, key=None):
    """Manual delineation of one HC-MS scan (He et al., "Retinal layer parcellation of optical coherence tomography
    images: data resource for multiple sclerosis and healthy controls"; reference ``Datasets.md:13``): a ``.mat`` file
    whose ``bd_pts`` holds the 9 boundary positions (pixels along the A-scan) as columns x B-scans x boundaries
    (1024 x 49 x 9).  Returns float32 ``[B-scans, boundaries, columns]`` -- the layout of BASELINE config 2 and of
    ``suite.boundary_metrics`` / ``suite.labels_from_boundaries``.  ``control_pts`` (the annotator's sparse control
    points, a cell array) is not needed for scoring and is ignored."""
    from scipy.io import loadmat
    mat = loadmat(path)
    names = [key] if key else ["bd_pts", "bds", "boundaries"]
    found = next((n for n in names if n in mat), None)
    if found is None:
        raise KeyError(f"{path}: none of {names} present (variables: {sorted(k for k in mat if not k.startswith('__'))})")
    bd = np.asarray(mat[found], dtype=np.float32)
    if bd.ndim != 3:
        raise ValueError(f"{path}: {found} has shape {bd.shape}, expected columns x B-scans x boundaries")
    return np.ascontiguousarray(np.transpose(bd, (1, 2, 0)))


def annotated_scans(layers, min_fraction=0.5):
    """Indices of the B-scans whose boundary rows are annotated in at least ``min_fraction`` of the columns
    (the Duke DME volumes annotate 11 of 61 B-scans)."""
    frac = np.isfinite(layers).all(axis=1).mean(axis=1)
    return np.nonzero(frac >= min_fraction)[0]


def read_labels(path, key=None):
    """uint8 label volume ``[slices, rows, cols]`` from ``.npy`` / ``.npz`` / ``.mhd``."""
    ext = os.path.splitext(path)[1].lower()
    if ext == ".npy":
        arr = np.load(path)
    elif ext == ".npz":
        with np.load(path) as z:
            arr = z[key if key else z.files[0]]
    elif ext == ".mhd":
        arr, _ = read_mhd(path)
    else:
        raise ValueError(f"unsupported label file {path}")
    if arr.ndim == 2:
        arr = arr[None]
    if arr.ndim != 3:
        raise ValueError(f"{path}: expected a 2-D or 3-D label array, got shape {arr.shape}")
    if arr.dtype != np.uint8:
        if arr.min() < 0 or arr.max() > 255:
            raise ValueError(f"{path}: labels outside [0, 255]")
        arr = arr.astype(np.uint8)
    return np.ascontiguousarray(arr)


def header_spacing_2d(true_path):
    """The B-scan pixel spacing ``(rows, cols)`` of a MetaImage label file: the last two axes of ``mhd_spacing``.
    ValueError for other formats and for a header without ``ElementSpacing``."""
    if os.path.splitext(true_path)[1].lower() != ".mhd":
        raise ValueError(f"{true_path}: spacing='header' needs a MetaImage (.mhd) file with ElementSpacing")
    _, header = read_mhd(true_path)
    try:
        sp = mhd_spacing(header)
    except KeyError:
        raise ValueError(f"{true_path}: the MetaImage header has no ElementSpacing") from None
    if len(sp) < 2:
        raise ValueError(f"{true_path}: ElementSpacing has {len(sp)} entry, a B-scan needs rows and columns")
    return sp[-2:]


def evaluate_files(true_path, pred_path, num_classes, *, spacing=None, **kwargs):
    """Score one predicted label volume against its ground truth, both on disk: reads the two files and runs
    ``suite.evaluate_host`` (chunked, copy/compute overlapped).  Keyword arguments go to ``evaluate_host``.
    ``spacing``: None (pixel units), ``(rows, cols)``, or ``"header"``: the ground truth's MetaImage ``ElementSpacing``
    (``header_spacing_2d``; ValueError for formats without one)."""
    from . import suite
    if isinstance(spacing, str):
        if spacing != "header":
            raise ValueError(f"spacing must be None, (rows, cols) or 'header', got {spacing!r}")
        spacing = header_spacing_2d(true_path)
    yt, yp = read_labels(true_path), read_labels(pred_path)
    if yt.shape != yp.shape:
        raise ValueError(f"shape mismatch: {yt.shape} vs {yp.shape}")
    return suite.evaluate_host(yt, yp, num_classes, spacing=spacing, **kwargs)
