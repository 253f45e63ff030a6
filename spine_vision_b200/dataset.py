"""``create_classification_dataset`` on the GPU path: the reference's public entry point
(``spine_vision/datasets/classification/__init__.py:122-235``) with the same configuration fields, output tree,
``annotations.csv`` columns and filesystem-resume semantics, but a different execution plan:

    reference (spider.py:90-178, phenikaa.py:142-226)        here
    ---------------------------------------------------     ---------------------------------------------------------
    for patient: for series:  read -> resample whole         1. walk the label files once -> list of SeriesJob (the same
      volume -> orient -> slice -> model (batch 1) ->           skip-if-all-levels-exist test, no pixels touched)
      5 x (crop -> PNG save) -> records                      2. per chunk of jobs: decode volumes on a thread pool into
                                                                pinned memory -> K0 -> K1 -> localizer -> K3 (one batch)
                                                             3. PNG-encode the chunk's crops on a thread pool, build records

Every numeric step is a kernel of ``libspine_b200.so`` (no CPU fallback); this module is the host logic around them
(label parsing, file naming, resume, CSV) and mirrors the reference's behaviour on bad input: a series whose reader
raises is skipped (spider.py:139-141, phenikaa.py:181-183).  Multi-GPU: pass ``rank`` / ``world_size`` to process every
``world_size``-th job; rank 0 writes the CSV after gathering the records (``gather_records``).
"""

from __future__ import annotations

import csv
import logging
import re
from dataclasses import dataclass, field
from pathlib import Path
from typing import Literal

import numpy as np
import torch
from pydantic import BaseModel, ConfigDict, computed_field

from . import hostio, ops, pipeline, volumes
from .cropping import LocalizationModel, load_localization_model

logger = logging.getLogger("spine_vision_b200.dataset")

CropMode = Literal["horizontal", "rotated"]
IVD_LEVEL_NAMES = ["L1/L2", "L2/L3", "L3/L4", "L4/L5", "L5/S1"]  # spider.py:181-182


# ------------------------------------------------------------------------------------------ public types (config.py, base.py)
class ClassificationDatasetConfig(BaseModel):
    """Field-for-field twin of the reference's ``ClassificationDatasetConfig`` (config.py:12-86; the three
    ``BaseConfig`` fields of core/config.py:8-15 included).  ``chunk_series``, ``io_threads`` and ``png_level`` are the
    only additions: how many series go through the GPU per batch and how wide the host decode / encode pools are."""

    model_config = ConfigDict(arbitrary_types_allowed=True, protected_namespaces=())

    verbose: bool = False
    enable_file_log: bool = False
    log_path: Path = Path.cwd() / "logs"

    base_path: Path = Path.cwd() / "data"
    output_name: str = "classification"
    localization_model_path: Path | None = None
    model_variant: Literal["tiny", "small", "base", "large", "xlarge", "v2_tiny", "v2_small", "v2_base", "v2_large", "v2_huge"] = "base"
    crop_size: tuple[int, int] = (256, 256)
    crop_delta_mm: tuple[float, float, float, float] = (55, 15, 17.5, 20)
    crop_mode: CropMode = "horizontal"
    last_disc_angle_boost: float = 1.0
    image_size: tuple[int, int] = (512, 512)
    include_phenikaa: bool = True
    include_spider: bool = True
    append_to_existing: bool = True
    device: str = "cuda:0"

    chunk_series: int = 128
    io_threads: int = 0
    png_level: int = 6

    @computed_field
    @property
    def phenikaa_path(self) -> Path:
        return self.base_path / "interim" / "Phenikaa"

    @computed_field
    @property
    def spider_path(self) -> Path:
        return self.base_path / "raw" / "SPIDER"

    @computed_field
    @property
    def output_path(self) -> Path:
        path = self.base_path / "processed" / self.output_name
        path.mkdir(parents=True, exist_ok=True)
        return path


class ClassificationRecord(BaseModel):
    """One row of ``annotations.csv`` (config.py:89-104): the 13 columns, in this order."""

    image_path: str
    patient_id: str
    ivd_level: int
    series_type: str
    source: str
    pfirrmann_grade: int
    disc_herniation: int
    disc_narrowing: int
    disc_bulging: int
    spondylolisthesis: int
    modic: int
    up_endplate: int
    low_endplate: int


@dataclass
class ProcessingResult:
    """datasets/base.py:10-24."""

    num_samples: int
    output_path: Path
    summary: str = ""


@dataclass
class ParsedImageInfo:
    """spider.py:185-193."""

    source: str
    patient_id: str
    series_type: str
    ivd_level: int
    filename: str


# ------------------------------------------------------------------------------------------ labels, names, resume
_NAME_RE = re.compile(r"^(phenikaa|spider)_(.+)_(sag_t[12])_L(\d)\.png$")  # spider.py:209


def parse_image_filename(filename: str) -> ParsedImageInfo | None:
    m = _NAME_RE.match(filename)
    if not m:
        return None
    return ParsedImageInfo(m.group(1), m.group(2), m.group(3), int(m.group(4)), filename)


def scan_existing_images(images_path: Path) -> list[ParsedImageInfo]:
    """The filesystem, not the CSV, says what is already done (spider.py:226-243)."""
    if not images_path.exists():
        return []
    found = (parse_image_filename(p.name) for p in images_path.glob("*.png"))
    return [f for f in found if f is not None]


def convert_spider_to_phenikaa_level(spider_level: int) -> int:
    """SPIDER counts from the sacrum (1 = L5/S1), the dataset from L1 (1 = L1/L2): spider.py:31-42."""
    return 6 - spider_level


def output_filename(source: str, patient_id, series_type: str, ivd_level: int) -> str:
    return f"{source}_{patient_id}_{series_type}_L{ivd_level}.png"


def _int(row: dict, key: str) -> int:
    return int(row.get(key, 0))


def make_record(source: str, filename: str, patient_id: str, ivd_level: int, series_type: str, row: dict) -> ClassificationRecord:
    """Label columns -> record.  SPIDER carries one ``Modic`` column (spider.py:160-175); Phenikaa carries one-hot
    ``Modic_0..3`` of which the first set one wins (phenikaa.py:88-93)."""
    if source == "phenikaa":
        modic = next((i for i in range(4) if row.get(f"Modic_{i}", "0") == "1"), 0)
    else:
        modic = _int(row, "Modic")
    return ClassificationRecord(
        image_path=f"images/{filename}", patient_id=str(patient_id), ivd_level=ivd_level, series_type=series_type, source=source,
        pfirrmann_grade=_int(row, "Pfirrman grade"), disc_herniation=_int(row, "Disc herniation"),
        disc_narrowing=_int(row, "Disc narrowing"), disc_bulging=_int(row, "Disc bulging"),
        spondylolisthesis=_int(row, "Spondylolisthesis"), modic=modic, up_endplate=_int(row, "UP endplate"),
        low_endplate=_int(row, "LOW endplate"))


def load_spider_labels(labels_path: Path) -> dict[int, dict[int, dict]]:
    """``radiological_gradings.csv`` -> patient -> dataset level -> row (spider.py:73-83)."""
    labels: dict[int, dict[int, dict]] = {}
    with open(labels_path, newline="") as f:
        for row in csv.DictReader(f):
            labels.setdefault(int(row["Patient"]), {})[convert_spider_to_phenikaa_level(int(row["IVD label"]))] = row
    return labels


def load_phenikaa_labels(labels_path: Path) -> dict[str, dict[int, dict]]:
    """``radiological_labels.csv`` -> patient -> level -> row (phenikaa.py:27-45)."""
    labels: dict[str, dict[int, dict]] = {}
    with open(labels_path, newline="") as f:
        for row in csv.DictReader(f):
            labels.setdefault(row["Patient ID"], {})[int(row["IVD label"])] = row
    return labels


def find_series_directory(patient_dir: Path, series_pattern: str) -> Path | None:
    """Case- and space-insensitive match of a series folder (phenikaa.py:48-65)."""
    want = series_pattern.lower().replace(" ", "")
    for sub in patient_dir.iterdir():
        if sub.is_dir() and sub.name.lower().replace(" ", "") == want:
            return sub
    return None


def recover_annotations(existing: list[ParsedImageInfo], spider_labels_path: Path, phenikaa_labels_path: Path):
    """Records for images already on disk, rebuilt from the source label files (recovery.py:40-160)."""
    out: dict[str, list[ClassificationRecord]] = {"phenikaa": [], "spider": []}
    if phenikaa_labels_path.exists():
        labels = load_phenikaa_labels(phenikaa_labels_path)
        for im in existing:
            row = labels.get(im.patient_id, {}).get(im.ivd_level) if im.source == "phenikaa" else None
            if row is not None:
                out["phenikaa"].append(make_record("phenikaa", im.filename, im.patient_id, im.ivd_level, im.series_type, row))
    else:
        logger.warning("Cannot recover Phenikaa annotations: %s not found", phenikaa_labels_path)
    if spider_labels_path.exists():
        slabels = load_spider_labels(spider_labels_path)
        for im in existing:
            if im.source != "spider":
                continue
            try:
                pid = int(im.patient_id)
            except ValueError:
                continue
            row = slabels.get(pid, {}).get(im.ivd_level)
            if row is not None:
                out["spider"].append(make_record("spider", im.filename, str(pid), im.ivd_level, im.series_type, row))
    else:
        logger.warning("Cannot recover SPIDER annotations: %s not found", spider_labels_path)
    return out["phenikaa"], out["spider"]


# ------------------------------------------------------------------------------------------ the work list
@dataclass
class SeriesJob:
    """One (patient, series) whose crops are still missing on disk."""

    source: str
    patient_id: str
    series_type: str
    path: Path  # .mha file (SPIDER) or series directory (Phenikaa)
    levels: dict[int, dict] = field(default_factory=dict)  # dataset level (1..5) -> label row, only the missing ones


def _missing_levels(source: str, patient_id, series_type: str, levels: dict[int, dict], existing: set[str]) -> dict[int, dict]:
    return {lvl: row for lvl, row in levels.items()
            if 1 <= lvl <= 5 and f"images/{output_filename(source, patient_id, series_type, lvl)}" not in existing}


def collect_spider_jobs(config: ClassificationDatasetConfig, existing: set[str]) -> list[SeriesJob]:
    """The iteration order and skip rules of ``process_spider`` (spider.py:62-108) without touching a pixel."""
    labels_path = config.spider_path / "radiological_gradings.csv"
    if not labels_path.exists():
        logger.warning("SPIDER labels not found: %s", labels_path)
        return []
    jobs = []
    for pid, levels in load_spider_labels(labels_path).items():
        for suffix, series_type in (("t1", "sag_t1"), ("t2", "sag_t2")):
            f = config.spider_path / "images" / f"{pid}_{suffix}.mha"
            if not f.exists():
                continue
            todo = _missing_levels("spider", pid, series_type, levels, existing)
            if todo:
                jobs.append(SeriesJob("spider", str(pid), series_type, f, todo))
    return jobs


def collect_phenikaa_jobs(config: ClassificationDatasetConfig, existing: set[str]) -> list[SeriesJob]:
    """``process_phenikaa`` (phenikaa.py:131-176) as a work list."""
    labels_path = config.phenikaa_path / "radiological_labels.csv"
    if not labels_path.exists():
        logger.warning("Phenikaa labels not found: %s", labels_path)
        return []
    jobs = []
    for pid, levels in load_phenikaa_labels(labels_path).items():
        pdir = config.phenikaa_path / "images" / pid
        if not pdir.exists():
            continue
        for pattern, series_type in (("sag t1", "sag_t1"), ("sag t2", "sag_t2")):
            sdir = find_series_directory(pdir, pattern)
            if sdir is None:
                continue
            todo = _missing_levels("phenikaa", pid, series_type, levels, existing)
            if todo:
                jobs.append(SeriesJob("phenikaa", pid, series_type, sdir, todo))
    return jobs


# ------------------------------------------------------------------------------------------ the batched body
def _read_chunk(jobs: list[SeriesJob], n_threads: int):
    """Decode a chunk of series.  MetaImage files go through the threaded native reader into pinned memory; anything
    else through ``hostio.read_medical_image`` (which raises for formats without a decoder -> the series is skipped)."""
    vols: list[hostio.MedicalVolume | None] = [None] * len(jobs)
    mha = [i for i, j in enumerate(jobs) if hostio.detect_format(j.path) in ("MHA", "MHD")]
    got, errs = hostio.read_volumes([jobs[i].path for i in mha], n_threads, midplane_only=True)  # the driver reads two slices per volume
    for k, i in enumerate(mha):
        vols[i] = got[k]
        if got[k] is None:
            logger.debug("Error processing %s: %s", jobs[i].path, errs[k])
    for i, j in enumerate(jobs):
        if i in mha:
            continue
        try:
            vols[i] = hostio.read_medical_image(j.path, midplane_only=True)
        except Exception as e:  # noqa: BLE001 -- spider.py:139-141 / phenikaa.py:181-183: any reader error skips the series
            logger.debug("Error reading %s: %s", j.path, e)
    return vols


def process_jobs(jobs: list[SeriesJob], config: ClassificationDatasetConfig, output_images_path: Path,
                 model: LocalizationModel | None) -> list[ClassificationRecord]:
    """Steps 2 and 3 of the module docstring for a list of jobs; returns the records of the crops written.

    A software pipeline over chunks of ``config.chunk_series`` series, so that neither the host nor the GPU waits for the other:

      read   (host thread)   decode chunk i+1 (native readers, only the two source planes K0 needs)
      A      (GPU, async)    chunk i: H2D of the source planes -> K0+K1 (fused) -> localizer; coordinates -> pinned host (async)
      B      (host + GPU)    chunk i-1: wait for ITS coordinates (the GPU is busy with A of chunk i meanwhile); rotated mode:
                             the exact host angle fit (np.polyfit, as the reference) -> K3 -> crops -> pinned host (async)
      C      (host thread)   chunk i-2: PNG encode + write, records

    Round 1 ran A..C of one chunk back to back with two blocking device->host reads (and, in rotated mode, a Python loop over
    the series between the localizer and K3): the GPU idled while the host worked."""
    from concurrent.futures import ThreadPoolExecutor

    records: list[ClassificationRecord] = []
    ch, cw = int(config.crop_size[0]), int(config.crop_size[1])
    step = max(1, config.chunk_series)
    chunks = [jobs[c0 : c0 + step] for c0 in range(0, len(jobs), step)]
    if not chunks:
        return records
    dev = torch.device(config.device)
    L = pipeline.NUM_LEVELS

    def stage_a(ci: int, chunk, vols):
        live = []
        for j, v in zip(chunk, vols):
            if v is None:
                continue
            if v.array.ndim != 3 or min(v.array.shape) < 1:
                logger.debug("Error processing %s: not a 3-D volume", j.path)
                continue
            try:
                volumes.lpi_axes(v.direction)
            except ValueError as e:
                logger.debug("Error processing %s: %s", j.path, e)
                continue
            live.append((j, v))
        if not live:
            return None
        n = len(live)
        pv = volumes.PinnedVolumes([v.array for _, v in live], [v.spacing for _, v in live], [v.direction for _, v in live],
                                   integer_pixels=[v.integer_pixels for _, v in live], pixel_kinds=[v.pixel_kind for _, v in live],
                                   cache_tag=f"dataset_slabs_{ci % 3}")  # three chunks are in flight at most
        pool = ops.SlicePool(torch.empty(max(pv.out_total, 4), dtype=torch.float32, device=dev),
                             torch.tensor(pv.out_offs, dtype=torch.int64).to(dev, non_blocking=True),
                             torch.tensor(pv.shapes, dtype=torch.int32).reshape(-1, 2).to(dev, non_blocking=True), list(pv.shapes),
                             h2d_bytes=pv.nbytes).set_pixel_kinds(pv.pixel_kinds)
        vols_d = pv.host.to(dev, non_blocking=True)
        desc_d = pv.chunk_descs(0, n).to(dev, non_blocking=True)
        if model is not None:
            planes = ops.midplane_normalize_resize(vols_d, desc_d, pool, config.image_size)
            coords = model.predict_u8(planes)
        else:
            ops.midplane_resample_into(vols_d, desc_d, pool)
            fb = pipeline.get_center_fallback_locations()  # Python floats in the reference, not model outputs: float64 for K3
            coords = torch.tensor([fb[i] for i in range(L)], dtype=torch.float64).unsqueeze(0).repeat(n, 1, 1).to(dev)
        coords_h = ops.PinnedCache.get(f"dataset_coords_{ci % 3}", n * L * 2, coords.dtype).view(n, L, 2)
        coords_h.copy_(coords, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return {"live": live, "pool": pool, "spacings": pv.spacings, "coords": coords, "coords_h": coords_h, "ev": ev, "ci": ci}

    def stage_b(st):
        if st is None:
            return None
        st["ev"].synchronize()  # this chunk's coordinates are on the host; the GPU is already working on the next chunk
        inv = None
        if config.crop_mode == "rotated":
            inv = pipeline.rotation_rows(st["coords_h"].numpy(), st["pool"].shapes, config.last_disc_angle_boost).pin_memory()
        crops, _, _ = pipeline.crop_levels(st["pool"], st["coords"], config.crop_delta_mm, st["spacings"], (ch, cw), None,
                                           mode=config.crop_mode, last_disc_angle_boost=config.last_disc_angle_boost, inv_affine=inv)
        n = len(st["live"])
        crops_h = ops.PinnedCache.get(f"dataset_crops_{st['ci'] % 3}", n * L * ch * cw, torch.uint8).view(n, L, ch, cw)
        crops_h.copy_(crops, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        st.update(crops=crops, crops_h=crops_h, ev=ev)
        return st

    with ThreadPoolExecutor(max_workers=2) as pool_io:
        pending_write = [None]

        def stage_c(st):
            if st is None:
                return
            st["ev"].synchronize()
            crops = st["crops_h"].numpy()  # [n, 5, ch, cw]
            sel, paths, recs = [], [], []
            for b, (j, _) in enumerate(st["live"]):
                for lvl, row in j.levels.items():
                    name = output_filename(j.source, j.patient_id, j.series_type, lvl)
                    sel.append((b, lvl - 1))
                    paths.append(output_images_path / name)
                    recs.append(make_record(j.source, name, j.patient_id, lvl, j.series_type, row))
            if sel:
                bi, li = zip(*sel)
                picked = crops[list(bi), list(li)]  # a copy: the pinned buffer is re-used three chunks later
                if pending_write[0] is not None:
                    pending_write[0].result()  # raises if a file of the previous chunk could not be written
                pending_write[0] = pool_io.submit(hostio.write_png_batch, picked, paths, config.png_level, config.io_threads)
                records.extend(recs)

        next_read = pool_io.submit(_read_chunk, chunks[0], config.io_threads)
        in_a = in_b = None  # the chunk whose stage A / stage B has been issued
        for ci in range(len(chunks) + 2):
            st_a = None
            if ci < len(chunks):
                vols = next_read.result()
                if ci + 1 < len(chunks):
                    next_read = pool_io.submit(_read_chunk, chunks[ci + 1], config.io_threads)
                st_a = stage_a(ci, chunks[ci], vols)
            st_b = stage_b(in_a)
            stage_c(in_b)
            in_a, in_b = st_a, st_b
        if pending_write[0] is not None:
            pending_write[0].result()
    return records


def process_spider(config, output_images_path: Path, model, existing_image_paths: set[str] | None = None):
    """Drop-in for ``process_spider`` (spider.py:45-178)."""
    return process_jobs(collect_spider_jobs(config, existing_image_paths or set()), config, output_images_path, model)


def process_phenikaa(config, output_images_path: Path, model, existing_image_paths: set[str] | None = None):
    """Drop-in for ``process_phenikaa`` (phenikaa.py:112-226)."""
    return process_jobs(collect_phenikaa_jobs(config, existing_image_paths or set()), config, output_images_path, model)


def gather_records(records: list[ClassificationRecord], group=None, failure: str | None = None):
    """All ranks' records on every rank, rank order (the per-rank order is the job order), and the failure messages of the
    ranks that could not finish their shard (so that every rank leaves the collective and raises the same error)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return records, ([failure] if failure else [])
    parts: list = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, {"records": [r.model_dump() for r in records], "failure": failure}, group=group)
    return ([ClassificationRecord(**d) for part in parts for d in part["records"]],
            [part["failure"] for part in parts if part["failure"]])


def write_annotations(csv_path: Path, records: list[ClassificationRecord]) -> None:
    """``annotations.csv`` exactly as the reference writes it (__init__.py:216-221)."""
    fieldnames = list(ClassificationRecord.model_fields.keys())
    with open(csv_path, "w", newline="") as f:
        writer = csv.DictWriter(f, fieldnames=fieldnames)
        writer.writeheader()
        for rec in records:
            writer.writerow(rec.model_dump())


def _plan_local(config, output_images_path: Path):
    """Everything that READS the output tree or the label files: resume scan (__init__.py:150-182), label recovery, job list."""
    existing = scan_existing_images(output_images_path)
    existing_paths: set[str] = set()
    recovered: list[ClassificationRecord] = []
    if existing and config.append_to_existing:
        logger.info("Found %d existing images on disk", len(existing))
        existing_paths = {f"images/{im.filename}" for im in existing}
        ph, sp = recover_annotations(existing, config.spider_path / "radiological_gradings.csv",
                                     config.phenikaa_path / "radiological_labels.csv")
        recovered = ph + sp
        orphans = len(existing) - len(recovered)
        if orphans > 0:
            logger.warning("%d existing images have no matching labels (labels may have been removed from source)", orphans)
    jobs: list[SeriesJob] = []
    if config.include_phenikaa:
        jobs += collect_phenikaa_jobs(config, existing_paths)
    if config.include_spider:
        jobs += collect_spider_jobs(config, existing_paths)
    return recovered, jobs


def plan_dataset(config, output_images_path: Path, rank: int = 0, world_size: int = 1):
    """(recovered records, job list).  Multi-rank: the plan is made ONCE, on rank 0, and broadcast.  If every rank scanned the
    tree itself, a late rank would see PNGs an early rank has already written, count them as existing and build a shorter job
    list -- the ``jobs[rank::world_size]`` shards would then disagree between ranks (series dropped or done twice, duplicate
    recovered rows)."""
    if world_size <= 1:
        return _plan_local(config, output_images_path)
    import torch.distributed as dist

    box = [_plan_local(config, output_images_path) if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    return box[0]


def create_classification_dataset(config: ClassificationDatasetConfig, rank: int = 0, world_size: int = 1) -> ProcessingResult:
    """Drop-in for ``create_classification_dataset`` (__init__.py:122-235).  With ``world_size > 1`` (one process per
    GPU, ``torch.distributed`` initialised) every rank takes every ``world_size``-th job, writes its own PNGs, and rank 0
    writes the CSV from the gathered records."""
    if config.verbose:
        logger.setLevel(logging.DEBUG)
    csv_path = config.output_path / "annotations.csv"
    output_images_path = config.output_path / "images"
    output_images_path.mkdir(parents=True, exist_ok=True)

    recovered, jobs = plan_dataset(config, output_images_path, rank, world_size)

    model: LocalizationModel | None = None
    failure: str | None = None
    new_records: list[ClassificationRecord] = []
    try:
        if config.localization_model_path is not None:
            logger.info("Loading localization model from: %s", config.localization_model_path)
            model = load_localization_model(config.localization_model_path, config.model_variant, config.device)
        else:
            logger.warning("No localization model provided, using center fallback locations")
        mine = jobs[rank::world_size] if world_size > 1 else jobs
        with torch.cuda.device(torch.device(config.device)):
            new_records = process_jobs(mine, config, output_images_path, model)
    except Exception as e:  # a failing rank must still meet the others in the gather below
        if world_size == 1:
            raise
        failure = f"rank {rank}: {type(e).__name__}: {e}"
        logger.error("dataset build failed on %s", failure)
    if world_size > 1:
        new_records, failures = gather_records(new_records, failure=failure)
        if failures:
            raise RuntimeError("create_classification_dataset failed on " + "; ".join(failures))

    all_records = recovered + new_records
    if rank == 0:
        write_annotations(csv_path, all_records)
    summary = (f"{len(all_records)} records ({len(recovered)} recovered, {len(new_records)} new) from "
               f"{len(jobs)} series; images: {output_images_path}; annotations: {csv_path}")
    logger.info(summary)
    return ProcessingResult(num_samples=len(all_records), output_path=config.output_path, summary=summary)
