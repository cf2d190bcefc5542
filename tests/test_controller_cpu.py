"""The N>1 host path on CPU (world_size-2, gloo): the single-box controller admits, orders, wires and
supervises replicas exactly as the reference operator would, and the job those replicas run
reproduces the committed golden losses of the reference-style gloo torchjob."""
import json
import os
import socket
import sys

import pytest

from torch_on_k8s_b200.controller import Controller
from torch_on_k8s_b200.sampler import ReplicaSampler

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def manifest(name, port, workers=1, queue=None, restart=None):
    c = {"name": "torch", "image": "local", "command": [sys.executable, os.path.join(HERE, "cpu_replica.py")],
         "ports": [{"name": "torchjob-port", "containerPort": port}]}
    m = {"metadata": {"name": name, "namespace": "default"},
         "spec": {"torchTaskSpecs": {"Master": {"template": {"spec": {"containers": [c]}}},
                                     "Worker": {"numTasks": workers,
                                                "template": {"spec": {"containers": [dict(c)]}}}}}}
    if queue:
        m["spec"]["schedulingPolicy"] = {"queue": queue}
    if restart:
        m["spec"]["torchTaskSpecs"]["Master"]["restartPolicy"] = restart
    return m


def test_mlp_torchjob_world2_matches_golden(tok_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("OUT_DIR", str(tmp_path))
    ctl = Controller(num_gpus=2, log_dir=str(tmp_path / "logs"), state_dir=str(tmp_path / "state"))
    uid = ctl.submit(manifest("mnist", free_port()))
    res = ctl.run_until_done(timeout=180)
    assert res[uid] == "Succeeded", (res, ctl.events[-5:])
    m = json.load(open(tmp_path / "mnist-master-0.json"))
    w = json.load(open(tmp_path / "mnist-worker-0.json"))
    assert (m["rank"], w["rank"], m["world"]) == (0, 1, 2)
    assert m["env"]["PYTHONUNBUFFERED"] == "0" and m["env"]["TOK8S_GPU"] != w["env"]["TOK8S_GPU"]
    gold = json.load(open(os.path.join(GOLD, "mlp_torchjob_n2", "run.json")))
    assert m["losses"] == pytest.approx(gold["losses"][:2], rel=0, abs=0)   # bit-identical floats
    reasons = [e[2] for e in ctl.events]
    assert reasons.index("JobEnqueued") < reasons.index("JobDequeued") < reasons.index("GangAdmitted")
    # DAG: the master is created before the worker
    pods = [e[3] for e in ctl.events if e[2] == "SuccessfulCreatePod"]
    assert pods[:2] == ["mnist-master-0", "mnist-worker-0"]
    st = ctl.jobs[uid].job.status
    assert st["taskStatuses"]["Master"]["succeed"] == 1 and st["taskStatuses"]["Worker"]["succeed"] == 1
    assert len(ctl.free_gpus) == 2
    # kubectl-shaped views (printer columns of torchjob_types.go:320-324)
    import io
    from torch_on_k8s_b200 import cli
    buf = io.StringIO()
    assert cli.cmd_get(str(tmp_path / "state"), out=buf) == 0
    lines = buf.getvalue().splitlines()
    assert lines[0].split() == ["NAME", "STATE", "AGE", "MODEL-VERSION", "MAX-LIFETIME", "TTL-AFTER-FINISHED"]
    assert lines[1].split()[:2] == ["mnist", "Succeeded"]
    buf = io.StringIO()
    assert cli.cmd_describe(str(tmp_path / "state"), "mnist", out=buf) == 0
    assert "JobSucceeded" in buf.getvalue() and "succeed=1" in buf.getvalue()
    assert cli.cmd_describe(str(tmp_path / "state"), "nope", out=io.StringIO()) == 1
    text = ctl.metrics.render()      # the reference's metric names (pkg/metrics/metrics.go)
    assert 'torch_on_k8s_jobs_created_total{kind="TorchJob"} 1.0' in text
    assert 'torch_on_k8s_jobs_successful_total{kind="TorchJob"} 1.0' in text
    assert "torch_on_k8s_jobs_all_pods_launch_delay_seconds_count" in text
    assert 'torch_on_k8s_tenant_queue_jobs_pending_count{queue="default"} 0.0' in text


def test_two_queued_jobs_gang_on_two_slots(tok_lib, tmp_path, monkeypatch):
    """BASELINE config 3 in miniature: two jobs of 2 replicas each on a 2-slot box — the second is
    held in its queue until the first releases its slots (all-or-nothing MinMember)."""
    monkeypatch.setenv("OUT_DIR", str(tmp_path))
    ctl = Controller(num_gpus=2)
    a = ctl.submit(manifest("ja", free_port(), queue="qa"))
    b = ctl.submit(manifest("jb", free_port(), queue="qb"))
    res = ctl.run_until_done(timeout=240)
    assert res == {a: "Succeeded", b: "Succeeded"}
    creates = [(e[0], e[3]) for e in ctl.events if e[2] == "SuccessfulCreatePod"]
    first = creates[0][1][:2]
    other = "jb" if first == "ja" else "ja"
    done_first = [e[0] for e in ctl.events if e[2] == "ExitedWithCode" and e[3].startswith(first)]
    start_other = [t for t, n in creates if n.startswith(other)]
    assert min(start_other) >= min(done_first)   # never more than 2 replicas on 2 slots


def test_failover_restarts_same_rank(tok_lib, tmp_path, monkeypatch):
    """Master exits 137 (SIGKILL, retryable under restartPolicy ExitCode): it is recreated with the
    same index => same RANK, the job goes through Restarting and still succeeds."""
    monkeypatch.setenv("OUT_DIR", str(tmp_path))
    monkeypatch.setenv("FAIL_ONCE", str(tmp_path / "failed.flag"))
    monkeypatch.setenv("FAIL_CODE", "137")
    ctl = Controller(num_gpus=2)
    uid = ctl.submit(manifest("fo", free_port()))
    res = ctl.run_until_done(timeout=240)
    reasons = [e[2] for e in ctl.events]
    assert "FailoverRecreate" in reasons
    assert res[uid] == "Succeeded", ctl.events[-6:]
    assert json.load(open(tmp_path / "fo-master-0.json"))["rank"] == 0


def test_permanent_exit_code_fails_job(tok_lib, tmp_path, monkeypatch):
    monkeypatch.setenv("OUT_DIR", str(tmp_path))
    monkeypatch.setenv("FAIL_ONCE", str(tmp_path / "failed.flag"))
    monkeypatch.setenv("FAIL_CODE", "1")      # permanent under ExitCode (failover.go:64-76)
    ctl = Controller(num_gpus=2)
    uid = ctl.submit(manifest("pf", free_port()))
    try:
        res = ctl.run_until_done(timeout=120)
        assert res[uid] == "Failed"
    finally:
        # cleanPodPolicy None keeps the worker, which would wait out gloo's 30-minute rendezvous
        # timeout for the failed master: stop it so that the test leaves no process behind
        for reps in ctl.jobs[uid].replicas.values():
            for r in reps.values():
                ctl._kill(r)


def test_replica_sampler_matches_distributed_sampler_goldens():
    cases = json.load(open(os.path.join(GOLD, "sampler.json")))
    for c in cases:
        for r in range(c["world"]):
            s = ReplicaSampler(c["n"], c["world"], r, shuffle=c["shuffle"], seed=c["seed"],
                               drop_last=c["drop_last"])
            s.set_epoch(c["epoch"])
            assert list(s) == c["indices"][r]          # bit-exact indices
    s = ReplicaSampler(100, 4, 1, seed=3)
    before = s.indices()
    s.reform(8, 5)
    t = ReplicaSampler(100, 8, 5, seed=3)
    assert s.indices() == t.indices() and s.indices() != before


def test_active_deadline_terminates_and_cleans_running_replicas(tok_lib, tmp_path, monkeypatch):
    """activeDurations (job.go:422-430) + cleanPodPolicy Running (:433-460): replicas that would run
    for 60 s are stopped after the 2 s deadline, the job is Failed "no longer active", slots free."""
    import time
    m = manifest("slow", free_port())
    for tt in ("Master", "Worker"):
        m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, "-c", "import time; time.sleep(60)"]
    m["spec"]["activeDurations"] = 2
    m["spec"]["clenPodPolicy"] = "Running"
    ctl = Controller(num_gpus=2)
    uid = ctl.submit(m)
    t0 = time.time()
    res = ctl.run_until_done(timeout=60)
    assert res[uid] == "Failed" and time.time() - t0 < 30
    assert any("no longer active" in e[3] for e in ctl.events if e[2] == "JobFailed")
    assert len(ctl.free_gpus) == 2
    assert all(r.proc.poll() is not None for reps in ctl.jobs[uid].replicas.values() for r in reps.values())


def test_torchelastic_loop_scales_workers_and_publishes_membership(tok_lib, tmp_path, monkeypatch):
    """a8 end to end on the host side: log scraping -> policy (min 1, max 2: rule 13 doubles after
    5 samples, then ReachMaxReplicas) -> a new worker replica is created, nobody is restarted, and
    the membership epoch file announces the new world."""
    monkeypatch.setenv("RUN_S", "7")
    m = manifest("el", free_port())
    for tt in ("Master", "Worker"):
        m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
    m["spec"]["enableTorchElastic"] = True
    m["spec"]["torchElasticPolicy"] = {"rendezvousBackend": "c10d", "rendezvousEndpoint": "x",
                                       "numMinReplicas": 1, "numMaxReplicas": 2}
    ctl = Controller(num_gpus=3, log_dir=str(tmp_path / "logs"), rdzv_dir=str(tmp_path),
                     elastic_period=0.25)
    uid = ctl.submit(m)
    res = ctl.run_until_done(timeout=90)
    assert res[uid] == "Succeeded", ctl.events[-8:]
    scale = [e for e in ctl.events if e[2] == "ElasticScale"]
    assert len(scale) == 1 and "Worker 1 -> 2" in scale[0][3]
    pods = [e[3] for e in ctl.events if e[2] == "SuccessfulCreatePod"]
    assert pods == ["el-master-0", "el-worker-0", "el-worker-1"]          # nobody was restarted
    members = [json.loads(e[3]) for e in ctl.events if e[2] == "MembershipPublished"]
    assert members[-1] == {"epoch": 1, "world": 3, "survivor_mask": 0b11,
                           "ranks": {"el-master-0": 0, "el-worker-0": 1, "el-worker-1": 2}}
    from torch_on_k8s_b200.worker import membership_update
    assert membership_update(members[-1], "el-worker-0", 0) == (3, 1, 0b11, 1)   # survivor re-forms
    assert membership_update(members[-1], "el-worker-1", 0) == (3, 2, 0b11, 1)   # joiner's view
    assert membership_update(members[-1], "el-worker-0", 1) is None              # already there
    assert membership_update(members[-1], "el-worker-9", 0) is None              # not a member
    st = ctl.jobs[uid].job.status["elasticScalingStatues"]["Worker"]
    assert st["elasticCondition"] == "ReachMaxReplicas" and st["curReplicas"] == 2
    # the torchrun args contract for the new size (SetClusterSpec :387-392)
    assert ctl.jobs[uid].job.cluster_spec("worker", 1)["env"][2] == {"name": "RANK", "value": "2"}


def test_torchelastic_revert_scales_in_and_deletes_out_of_range_replica(tok_lib, tmp_path, monkeypatch):
    """Scale-out that makes the per-replica latency worse is reverted (rule 12, ReachMaxMetric): the
    out-of-range replica is deleted (reconcileOnePod, pod.go:648-651), its GPU slot freed, the
    survivors keep running, and a second membership epoch announces the smaller world."""
    monkeypatch.setenv("RUN_S", "8")
    monkeypatch.setenv("ADAPTIVE", "1")
    m = manifest("si", free_port())
    for tt in ("Master", "Worker"):
        m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
    m["spec"]["enableTorchElastic"] = True
    m["spec"]["torchElasticPolicy"] = {"rendezvousBackend": "c10d", "rendezvousEndpoint": "x",
                                       "numMinReplicas": 1, "numMaxReplicas": 2}
    ctl = Controller(num_gpus=3, rdzv_dir=str(tmp_path), log_dir=str(tmp_path / "logs"),
                     elastic_period=0.25)
    uid = ctl.submit(m)
    res = ctl.run_until_done(timeout=90)
    assert res[uid] == "Succeeded", ctl.events[-8:]
    scale = [e[3] for e in ctl.events if e[2] == "ElasticScale"]
    assert len(scale) == 2 and "scale: Worker 1 -> 2" in scale[0] and "revert: Worker 2 -> 1" in scale[1]
    assert [e[3] for e in ctl.events if e[2] == "SuccessfulDeletePod"] == ["si-worker-1"]
    members = [json.loads(e[3]) for e in ctl.events if e[2] == "MembershipPublished"]
    assert [(d["epoch"], d["world"], d["survivor_mask"]) for d in members] == [(1, 3, 0b11), (2, 2, 0b011)]
    assert ctl.jobs[uid].job.num_tasks("Worker") == 1 and len(ctl.free_gpus) == 3
    st = ctl.jobs[uid].job.status["elasticScalingStatues"]["Worker"]
    assert st["elasticCondition"] == "Stop" and st["curReplicas"] == 1 and st["lastReplicas"] == 2


def test_scale_request_publishes_membership_only_when_every_replica_runs(tok_lib, tmp_path, monkeypatch):
    """Row a7, user-driven: Controller.scale() edits Worker.numTasks on a running job; the reconcile
    creates the replicas it has GPUs for.  With one GPU short the new membership is NOT announced
    (survivors re-forming towards a Pending replica would block in the rendezvous); after scaling back
    to a size that fits, the out-of-range replicas are deleted and nothing that equals the already
    known membership is re-announced; a scale-out that fits is announced once, nobody restarts."""
    monkeypatch.setenv("RUN_S", "8")
    m = manifest("sc", free_port())
    for tt in ("Master", "Worker"):
        m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
    ctl = Controller(num_gpus=3, rdzv_dir=str(tmp_path), log_dir=str(tmp_path / "logs"))
    uid = ctl.submit(m)
    import time
    t0 = time.time()
    while time.time() - t0 < 20 and ctl.jobs[uid].job.last_condition() != "Running":
        ctl.tick()
        time.sleep(0.05)
    assert ctl.jobs[uid].job.last_condition() == "Running"
    with pytest.raises(ValueError):
        ctl.scale(uid, "Worker", 8)                       # 1 master + 8 workers > 8 replicas
    assert ctl.scale(uid, "Worker", 3) == 1               # needs 4 GPUs, the box has 3
    for _ in range(10):
        ctl.tick()
        time.sleep(0.05)
    reps = ctl.jobs[uid].replicas["Worker"]
    assert sorted(reps) == [0, 1, 2] and reps[2].proc is None and reps[2].phase == "Pending"
    assert not [e for e in ctl.events if e[2] == "MembershipPublished"]
    assert ctl.scale(uid, "Worker", 2) == 2               # fits: worker-2 (Pending) goes away
    for _ in range(10):
        ctl.tick()
        time.sleep(0.05)
    members = [json.loads(e[3]) for e in ctl.events if e[2] == "MembershipPublished"]
    assert members == [{"epoch": 2, "world": 3, "survivor_mask": 0b011,
                        "ranks": {"sc-master-0": 0, "sc-worker-0": 1, "sc-worker-1": 2}}]
    assert ctl.scale(uid, "Worker", 1) == 3
    res = ctl.run_until_done(timeout=60)
    assert res[uid] == "Succeeded", ctl.events[-8:]
    members = [json.loads(e[3]) for e in ctl.events if e[2] == "MembershipPublished"]
    assert (members[-1]["epoch"], members[-1]["world"], members[-1]["survivor_mask"]) == (3, 2, 0b011)
    pods = [e[3] for e in ctl.events if e[2] == "SuccessfulCreatePod"]
    assert pods == ["sc-master-0", "sc-worker-0", "sc-worker-1"]     # survivors were never restarted
    assert len(ctl.free_gpus) == 3


def test_full_box_keeps_low_priority_job_queued_so_priority_wins(tok_lib, tmp_path, monkeypatch):
    """Quota filter sees real GPU usage (quota.go:97-131): while job a holds every GPU, job b (other
    tenant, same default quota) is NOT dequeued; a high-priority job c that arrives later in b's queue
    is therefore admitted before b once a finishes."""
    monkeypatch.setenv("RUN_S", "3")

    def mk(name, queue, prio=None):
        m = manifest(name, free_port(), queue=queue)
        for tt in ("Master", "Worker"):
            m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
                [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
        if prio is not None:
            m["spec"].setdefault("schedulingPolicy", {})["priority"] = prio
        return m
    ctl = Controller(num_gpus=2, rdzv_dir=str(tmp_path))
    a = ctl.submit(mk("qa", "team-a"))
    import time
    t0 = time.time()
    while time.time() - t0 < 20 and len(ctl.free_gpus) > 0:
        ctl.tick()
        time.sleep(0.05)
    assert len(ctl.free_gpus) == 0
    b = ctl.submit(mk("qb", "team-b", prio=1))
    for _ in range(12):
        ctl.tick()
        time.sleep(0.05)
    assert not ctl.jobs[b].dequeued                      # the box is full: b waits in its queue
    c = ctl.submit(mk("qc", "team-b", prio=100))
    res = ctl.run_until_done(timeout=90)
    assert set(res.values()) == {"Succeeded"}, res
    order = [e[1] for e in ctl.events if e[2] == "JobDequeued"]
    assert order == [a, c, b]


def test_metrics_endpoint_and_replica_telemetry(tok_lib, tmp_path):
    """f3: the reference's metric names over GET /metrics (main.go:59), and the two new series fed
    from `TOK8S_METRIC {...}` lines a replica prints (worker.report_metric) — scraped like the
    torchelastic progress line."""
    import urllib.request
    from torch_on_k8s_b200.controller import ManagedJob, ReplicaProc
    from torch_on_k8s_b200.job import TorchJob
    ctl = Controller(num_gpus=2)
    log = tmp_path / "j-master-0.log"
    log.write_text('noise\nTOK8S_METRIC {"busbw_gbps": 512.5}\nTOK8S_METRIC {"reform_s": 0.25}\nTOK8S_METRIC {"half')
    job = TorchJob(manifest("j", free_port()))
    mj = ManagedJob(job=job, uid="default/j")
    mj.replicas["Master"] = {0: ReplicaProc("Master", 0, 0, log_path=str(log))}
    ctl._scrape_metrics(mj)
    ctl._scrape_metrics(mj)                       # nothing is counted twice; the partial line waits
    port = free_port()
    ctl.metrics.serve(port)
    text = urllib.request.urlopen("http://127.0.0.1:%d/metrics" % port, timeout=10).read().decode()
    assert 'torch_on_k8s_allreduce_busbw_gbps{job="j"} 512.5' in text
    assert 'torch_on_k8s_reform_latency_seconds_count{job="j"} 1.0' in text
    assert "torch_on_k8s_jobs_created_total" in text and "torch_on_k8s_tenant_queue_jobs_pending_count" in text


def test_joiner_waits_for_the_membership_that_lists_it(tmp_path):
    """A replica started into a running job joins at the epoch the controller ANNOUNCES (not the one
    it was started at): it waits for the first document with epoch >= its own that lists it; a
    membership that never lists it (a reverted scale-out) times out instead of joining a wrong group."""
    import threading
    import time
    from torch_on_k8s_b200.worker import membership_update, wait_for_membership
    rdzv = str(tmp_path / "tok8s-j-1")

    def publish(doc, delay):
        time.sleep(delay)
        with open(rdzv + ".members.tmp", "w") as f:
            json.dump(doc, f)
        os.replace(rdzv + ".members.tmp", rdzv + ".members")
    with open(rdzv + ".members", "w") as f:     # an older membership without the joiner
        json.dump({"epoch": 1, "world": 2, "ranks": {"j-master-0": 0, "j-worker-0": 1}}, f)
    doc3 = {"epoch": 3, "world": 3, "survivor_mask": 3,
            "ranks": {"j-master-0": 0, "j-worker-0": 1, "j-worker-1": 2}}
    threading.Thread(target=publish, args=(doc3, 0.3), daemon=True).start()
    assert wait_for_membership(rdzv, "j-worker-1", 2, timeout_s=10) == (2, 3, 3)
    with pytest.raises(TimeoutError):
        wait_for_membership(rdzv, "j-worker-9", 2, timeout_s=0.3)
    assert membership_update(doc3, "j-worker-0", 1) == (3, 1, 3, 3)     # survivor's step
    assert membership_update(doc3, "j-worker-0", 3) is None             # already at that epoch


def test_scale_in_drains_replicas_gracefully(tok_lib, tmp_path, monkeypatch):
    """In-place scale-in: the replicas that fall out of [0, numTasks) are NOT killed on the spot (their
    peers would find them dead in the middle of a gradient exchange): they are dropped from the
    published membership first, leave on their own at a step boundary, and only then does the
    controller reap them and free their GPU slots; one that overstays drain_grace_s is deleted the
    reference's way (reconcileOnePod, pod.go:648-651)."""
    import time
    monkeypatch.setenv("RUN_S", "30")
    monkeypatch.setenv("EXIT_WHEN_DROPPED", "1")
    m = manifest("dr", free_port(), workers=2)
    for tt in ("Master", "Worker"):
        m["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
    ctl = Controller(num_gpus=3, rdzv_dir=str(tmp_path), log_dir=str(tmp_path / "logs"),
                     drain_grace_s=20)
    uid = ctl.submit(m)
    t0 = time.time()
    while time.time() - t0 < 20 and ctl.jobs[uid].job.last_condition() != "Running":
        ctl.tick()
        time.sleep(0.05)
    assert len(ctl.free_gpus) == 0
    assert ctl.scale(uid, "Worker", 1) == 1
    t1 = time.time()
    while time.time() - t1 < 15 and not any(e[2] == "SuccessfulDeletePod" for e in ctl.events):
        ctl.tick()
        time.sleep(0.05)
    took = time.time() - t1
    order = [e[2] for e in ctl.events if e[2] in ("DrainingPod", "MembershipPublished", "SuccessfulDeletePod")]
    assert order == ["DrainingPod", "MembershipPublished", "SuccessfulDeletePod"]
    assert took < 10                                    # it left by itself, long before the grace period
    doc = [json.loads(e[3]) for e in ctl.events if e[2] == "MembershipPublished"][-1]
    assert doc == {"epoch": 1, "world": 2, "survivor_mask": 0b011,
                   "ranks": {"dr-master-0": 0, "dr-worker-0": 1}}
    assert len(ctl.free_gpus) == 1 and "Worker" in ctl.jobs[uid].replicas and \
        sorted(ctl.jobs[uid].replicas["Worker"]) == [0]
    # a replica that does not leave is deleted when the grace period is over
    monkeypatch.delenv("EXIT_WHEN_DROPPED")
    ctl2 = Controller(num_gpus=3, rdzv_dir=str(tmp_path / "b"), drain_grace_s=1.0)
    os.makedirs(tmp_path / "b", exist_ok=True)
    m2 = manifest("dr2", free_port(), workers=2)
    for tt in ("Master", "Worker"):
        m2["spec"]["torchTaskSpecs"][tt]["template"]["spec"]["containers"][0]["command"] = \
            [sys.executable, os.path.join(HERE, "cpu_elastic_replica.py")]
    uid2 = ctl2.submit(m2)
    t0 = time.time()
    while time.time() - t0 < 20 and ctl2.jobs[uid2].job.last_condition() != "Running":
        ctl2.tick()
        time.sleep(0.05)
    ctl2.scale(uid2, "Worker", 1)
    t1 = time.time()
    while time.time() - t1 < 15 and not any(e[2] == "SuccessfulDeletePod" for e in ctl2.events):
        ctl2.tick()
        time.sleep(0.05)
    assert 0.9 <= time.time() - t1 < 10 and len(ctl2.free_gpus) == 1
    for c in (ctl, ctl2):
        for mj in c.jobs.values():
            for reps in mj.replicas.values():
                for r in reps.values():
                    c._kill(r)
