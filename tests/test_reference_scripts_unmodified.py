"""The reference's OWN scripts, byte for byte, running on this framework through the ``tensorflow`` drop-in shim
(``distributed_tensorflow_b200/compat``): the strongest parity check available without TensorFlow -- every symbol,
default, device string and hook protocol the scripts exercise has to behave (SURVEY section 2.2, A1-A23).

The scripts are not part of this repository: those tests need a checkout of the reference project, named by
``DTF_REFERENCE_DIR``, and skip without one.  The scripts hard-code ``localhost:2222-2224`` / explicit host flags, so these
tests must not run concurrently with each other."""
import os
import subprocess
import sys
import time

import pytest

REF = os.environ.get("DTF_REFERENCE_DIR", "/root/reference")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not os.path.exists(os.path.join(REF, "distributed_mnist.py")),
                                     reason="reference checkout not available")


def _env(tmp_path):
    e = dict(os.environ, CUDA_VISIBLE_DEVICES="", DTF_HDFS_ROOT=str(tmp_path / "hdfs"))
    e["PYTHONPATH"] = ROOT + os.pathsep + e.get("PYTHONPATH", "")
    return e


def _cmd(script, *args):
    return [sys.executable, "-u", "-m", "distributed_tensorflow_b200.compat.run", os.path.join(REF, script)] + list(args)


def _run(tmp_path, script, *args, timeout=300):
    r = subprocess.run(_cmd(script, *args), capture_output=True, text=True, timeout=timeout, env=_env(tmp_path), cwd=str(tmp_path))
    assert r.returncode == 0, "exit %d\n%s\n%s" % (r.returncode, r.stdout[-3000:], r.stderr[-3000:])
    return r.stdout


class _Tasks:
    """Background tasks (ps / serving workers) that are terminated when the block ends."""

    def __init__(self, tmp_path):
        self.tmp_path, self.procs = tmp_path, []

    def start(self, script, *args):
        log = open(self.tmp_path / ("task%d.log" % len(self.procs)), "w")
        # a background task that is ALSO a client (every worker of example_distributed_server.py) keeps serving after its own run
        # is done, until the block ends: the foreground task's success must not depend on which of the two finishes first
        env = dict(_env(self.tmp_path), DTF_EXIT_SERVE_S="300")
        self.procs.append(subprocess.Popen(_cmd(script, *args), stdout=log, stderr=subprocess.STDOUT, env=env, cwd=str(self.tmp_path)))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for p in self.procs:
            p.terminate()
        for p in self.procs:
            try:
                p.wait(timeout=10)
            except subprocess.TimeoutExpired:
                p.kill()


def _golden(out):
    flat = out.replace("\n", " ")
    for v in ("9.", "21.", "33.", "45."):
        assert v in flat, out


@needs_reference
def test_reference_standalone_py(tmp_path):
    out = _run(tmp_path, "standalone.py", timeout=600)           # 10 000 tower steps on one fixed batch
    assert "affine_last/w" in out and "GPU" in out               # '2块GPU用时: ...s'


@needs_reference
def test_reference_example_in_graph_py(tmp_path):
    with _Tasks(tmp_path) as t:
        t.start("example_in_graph.py", "--job_name=ps", "--task_index=0")
        t.start("example_in_graph.py", "--job_name=worker", "--task_index=1")
        time.sleep(1.0)
        _golden(_run(tmp_path, "example_in_graph.py", "--job_name=worker", "--task_index=0", timeout=120))
    assert (tmp_path / "timeline_client.json").exists() and (tmp_path / "logs").exists()


@needs_reference
def test_reference_distributed_server_and_client_py(tmp_path):
    with _Tasks(tmp_path) as t:
        t.start("example_distributed_server.py", "--job_name=ps", "--task_index=0")
        t.start("example_distributed_server.py", "--job_name=worker", "--task_index=1")
        time.sleep(1.0)
        _golden(_run(tmp_path, "example_distributed_server.py", "--job_name=worker", "--task_index=0", timeout=120))
    # the pure client needs worker 0 up as well: serve-only tasks from this repo's twin of the server script
    serve = [sys.executable, "-u", os.path.join(ROOT, "examples", "example_distributed_server.py")]
    procs = [subprocess.Popen(serve + ["--job_name=%s" % j, "--task_index=%d" % i], env=_env(tmp_path), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for j, i in (("ps", 0), ("worker", 0), ("worker", 1))]
    try:
        for p in procs:
            assert "serving" in p.stdout.readline()
        _golden(_run(tmp_path, "example_distributed_client.py", timeout=120))
    finally:
        for p in procs:
            p.terminate()
        for p in procs:
            p.wait(timeout=10)


@needs_reference
@pytest.mark.parametrize("sync", [True, False])
def test_reference_example_between_graph_py(tmp_path, sync):
    hosts = ["--ps_hosts=127.0.0.1:22251", "--worker_hosts=127.0.0.1:22252,127.0.0.1:22253"]
    mode = ["--is_sync=%s" % sync]
    with _Tasks(tmp_path) as t:
        t.start("example_between_graph.py", "--job_name=ps", "--task_index=0", *hosts)
        t.start("example_between_graph.py", "--job_name=worker", "--task_index=1", *(hosts + mode))
        out = _run(tmp_path, "example_between_graph.py", "--job_name=worker", "--task_index=0", *(hosts + mode), timeout=400)
    last = [l for l in out.splitlines() if "weight:" in l][-1]
    w = float(last.split("weight:")[1].split(",")[0])
    b = float(last.split("biase:")[1].split(",")[0])
    assert abs(w - 2.0) < 0.1 and abs(b - 10.0) < 0.2, last       # y = 2x + 10 recovered (example_between_graph.py:36)
    assert (tmp_path / "hdfs" / "test" / "ckpt" / "checkpoint").exists()      # hdfs:// checkpoint dir mapped to a local root


@needs_reference
@pytest.mark.skipif(os.environ.get("DTF_SLOW_TESTS", "0") != "1", reason="10 000 global steps (~2 min): DTF_SLOW_TESTS=1")
def test_reference_distributed_mnist_then_predict_py(tmp_path):
    hosts = ["--ps_hosts=127.0.0.1:22221", "--worker_hosts=127.0.0.1:22222,127.0.0.1:22223"]
    with _Tasks(tmp_path) as t:
        t.start("distributed_mnist.py", "--job_name=ps", "--task_index=0", *hosts)
        t.start("distributed_mnist.py", "--job_name=worker", "--task_index=1", "--issync=True", *hosts)
        out = _run(tmp_path, "distributed_mnist.py", "--job_name=worker", "--task_index=0", "--issync=True", *hosts, timeout=1500)
    assert "Training elapsed time" in out and "global step:" in out
    pred = _run(tmp_path, "distributed_mnist_predict.py", timeout=300)
    nums = [int(x) for x in pred.split() if x.isdigit()]
    assert nums and nums[-1] > 4500, pred            # > 90 % of the 5 000 validation images


@pytest.mark.parametrize("sync", ["False", "True"])
def test_tf_style_supervisor_program_through_the_shim(tmp_path, sync):
    """A ``tf.app.run`` / ``tf.train.Supervisor`` / chief-queue-runner program in TF spelling (tests/fixtures) on
    1 ps + 2 workers: the generation of scripts the reference descends from (``distributed_mnist.py:57``)."""
    import re
    script = os.path.join(ROOT, "tests", "fixtures", "tf_style_replica.py")
    hosts = ["--ps_hosts=127.0.0.1:22281", "--worker_hosts=127.0.0.1:22282,127.0.0.1:22283", "--sync_replicas=%s" % sync]

    def cmd(job, idx):
        return [sys.executable, "-u", "-m", "distributed_tensorflow_b200.compat.run", script, "--job_name=%s" % job,
                "--task_index=%d" % idx] + hosts
    procs = [subprocess.Popen(cmd("ps", 0), env=_env(tmp_path), cwd=str(tmp_path), stdout=subprocess.DEVNULL, stderr=subprocess.STDOUT)]
    logs = []
    try:
        for i in (0, 1):
            f = open(tmp_path / ("w%d.log" % i), "w")
            logs.append(f)
            procs.append(subprocess.Popen(cmd("worker", i), env=_env(tmp_path), cwd=str(tmp_path), stdout=f, stderr=subprocess.STDOUT))
        for p in procs[1:]:
            assert p.wait(timeout=300) == 0, open(tmp_path / "w0.log").read()[-2000:] + open(tmp_path / "w1.log").read()[-2000:]
    finally:
        for p in procs:
            if p.poll() is None:
                p.kill()
        for f in logs:
            f.close()
    for i in (0, 1):
        out = open(tmp_path / ("w%d.log" % i)).read()
        assert "Session initialization complete." in out
        val = float(re.findall(r"validation cross entropy = ([0-9][0-9.eE+-]*)", out)[-1])
        assert val < 5000.0                                         # ~11500 for the untrained model (5000 images, batch sum)
