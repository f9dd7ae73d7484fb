#include <faabric/batch-scheduler/BatchScheduler.h>
#include <faabric/executor/Executor.h>
#include <faabric/executor/ExecutorFactory.h>
#include <faabric/scheduler/FunctionCallClient.h>
#include <faabric/scheduler/Scheduler.h>
#include <faabric/snapshot/SnapshotClient.h>
#include <faabric/transport/common.h>
#include <faabric/util/batch.h>
#include <faabric/util/environment.h>
#include <faabric/util/func.h>
#include <faabric/util/logging.h>
#include <faabric/util/testing.h>

namespace faabric::scheduler {

Scheduler& getScheduler()
{
    static Scheduler sch;
    return sch;
}

Scheduler::Scheduler()
  : thisHost(faabric::transport::getThisHostAddress())
  , conf(faabric::util::getSystemConfig())
  , reg(faabric::snapshot::getSnapshotRegistry())
  , broker(faabric::transport::getPointToPointBroker())
{
    // Idle executors are reaped periodically
    if (conf.reaperIntervalSeconds > 0) {
        reaperThread.start(conf.reaperIntervalSeconds);
    }
}

Scheduler::~Scheduler()
{
    if (!_isShutdown) {
        SPDLOG_DEBUG("Destructing scheduler without shutting down first");
    }
    reaperThread.stop();
    keepAliveThread.stop();
}

std::string Scheduler::getThisHost()
{
    return thisHost;
}

// ---------------------------------------------------------------------------
// Membership
// ---------------------------------------------------------------------------
void Scheduler::addHostToGlobalSet(
  const std::string& hostIp,
  std::shared_ptr<faabric::HostResources> overwriteResources)
{
    auto req = std::make_shared<faabric::planner::RegisterHostRequest>();
    req->mutable_host()->set_ip(hostIp);
    req->set_overwrite(false);
    if (overwriteResources != nullptr) {
        req->mutable_host()->set_slots(overwriteResources->slots());
        req->mutable_host()->set_usedslots(overwriteResources->usedslots());
        req->set_overwrite(true);
    } else if (hostIp == thisHost) {
        // Execution slots: CPU cores, or slots-per-GPU x GPUs on a GPU box.
        // OVERRIDE_CPU_COUNT wins on both, as it also sizes the executor's
        // thread pool
        int gpus = faabric::util::getUsableGpus();
        int slots = (conf.overrideCpuCount > 0 || gpus == 0) ? (int)faabric::util::getUsableCores()
                                                             : gpus * conf.slotsPerGpu;
        req->mutable_host()->set_slots(slots);
        req->mutable_host()->set_usedslots(0);
    }
    int plannerTimeout = faabric::planner::getPlannerClient().registerHost(req);
    // Keep-alive at half the planner's timeout for every host this process
    // serves: itself and the per-GPU virtual hosts aliased to it
    const bool servedHere = hostIp == thisHost || faabric::transport::resolveHostAlias(hostIp) != hostIp;
    if (servedHere) {
        servedHosts.insert(hostIp);
    }
    if (servedHere && !faabric::util::isTestMode()) {
        keepAliveThread.setRequest(req);
        if (!keepAliveRunning) {
            keepAliveThread.startMs(std::max(100, plannerTimeout * 1000 / 2));
            keepAliveRunning = true;
        }
    }
}

void Scheduler::addHostToGlobalSet()
{
    addHostToGlobalSet(thisHost);
}

void Scheduler::removeHostFromGlobalSet(const std::string& hostIp)
{
    auto req = std::make_shared<faabric::planner::RemoveHostRequest>();
    servedHosts.erase(hostIp);
    if (keepAliveRunning && keepAliveThread.removeRequest(hostIp) == 0) {
        keepAliveThread.stop();
        keepAliveRunning = false;
    }
    req->mutable_host()->set_ip(hostIp);
    faabric::planner::getPlannerClient().removeHost(req);
}

void Scheduler::setThisHostResources(faabric::HostResources& res)
{
    addHostToGlobalSet(thisHost, std::make_shared<faabric::HostResources>(res));
    conf.overrideCpuCount = res.slots();
}

// ---------------------------------------------------------------------------
// Lifecycle
// ---------------------------------------------------------------------------
void Scheduler::resetThreadLocalCache()
{
    clearFunctionCallClients();
    faabric::snapshot::clearSnapshotClients();
}

void Scheduler::reset()
{
    SPDLOG_DEBUG("Resetting scheduler");
    resetThreadLocalCache();
    // Shut the executors down outside the lock: their threads may call back
    std::vector<std::shared_ptr<faabric::executor::Executor>> toStop;
    {
        std::unique_lock<std::shared_mutex> lock(mx);
        for (auto& [key, vec] : executors) {
            for (auto& e : vec) {
                toStop.push_back(e);
            }
        }
        executors.clear();
    }
    {
        std::lock_guard<IdleLock> lk(idleMx);
        idleExecutors.clear();
    }
    for (auto& e : toStop) {
        e->shutdown();
    }
    {
        std::lock_guard<std::mutex> lk(threadResultsMx);
        threadResultMessages.clear();
    }
    {
        std::unique_lock<std::shared_mutex> lock(mx);
        recordedMessages.clear();
    }
    faabric::planner::getPlannerClient().clearCache();
    _isShutdown = false;
}

void Scheduler::shutdown()
{
    reset();
    reaperThread.stop();
    // No more keep-alives, then withdraw every host this process served
    if (keepAliveRunning) {
        keepAliveThread.stop();
        keepAliveRunning = false;
    }
    std::set<std::string> hosts = servedHosts;
    hosts.insert(thisHost);
    for (const auto& h : hosts) {
        try {
            removeHostFromGlobalSet(h);
        } catch (const std::exception& e) {
            SPDLOG_DEBUG("Could not deregister host {} on shutdown: {}", h, e.what());
        }
    }
    servedHosts.clear();
    _isShutdown = true;
}

void SchedulerReaperThread::doWork()
{
    getScheduler().reapStaleExecutors();
}

void Scheduler::notifyExecutorIdle(const std::string& funcKey, std::weak_ptr<faabric::executor::Executor> executor)
{
    std::lock_guard<IdleLock> lk(idleMx);
    idleExecutors[funcKey].push_back(std::move(executor));
}

int Scheduler::reapStaleExecutors()
{
    std::unique_lock<std::shared_mutex> lock(mx);
    if (executors.empty()) {
        return 0;
    }
    int reaped = 0;
    std::vector<std::shared_ptr<faabric::executor::Executor>> toStop;
    for (auto it = executors.begin(); it != executors.end();) {
        auto& vec = it->second;
        for (auto e = vec.begin(); e != vec.end();) {
            long idle = (*e)->getMillisSinceLastExec();
            if (idle < conf.boundTimeout || (*e)->isExecuting()) {
                ++e;
                continue;
            }
            // Only reap what we can claim (not mid-way through being claimed)
            if (!(*e)->tryClaim()) {
                ++e;
                continue;
            }
            SPDLOG_DEBUG("Reaping stale executor {} ({}ms idle)", (*e)->id, idle);
            toStop.push_back(*e);
            e = vec.erase(e);
            reaped++;
        }
        if (vec.empty()) {
            it = executors.erase(it);
        } else {
            ++it;
        }
    }
    lock.unlock();
    for (auto& e : toStop) {
        e->shutdown();
    }
    return reaped;
}

long Scheduler::getFunctionExecutorCount(const faabric::Message& msg)
{
    std::shared_lock<std::shared_mutex> lock(mx);
    long n = 0;
    std::string prefix = faabric::util::funcToString(msg, false);
    for (const auto& [key, vec] : executors) {
        if (key == prefix || key.rfind(prefix + ":", 0) == 0 || key.rfind(prefix + "@", 0) == 0) {
            n += (long)vec.size();
        }
    }
    return n;
}

void Scheduler::flushLocally()
{
    SPDLOG_INFO("Flushing host {}", thisHost);
    reset();
    faabric::executor::getExecutorFactory()->flushHost();
}

// ---------------------------------------------------------------------------
// Execution
// ---------------------------------------------------------------------------
std::string Scheduler::executorKeyFor(const faabric::Message& msg)
{
    // Executors are warm per user/function and reused across apps.  One
    // scheduler may serve several per-GPU virtual hosts: an executor is bound
    // to the GPU of the host it was created for, so the host is part of the key
    std::string key = faabric::util::funcToString(msg, false);
    if (!msg.executedhost().empty() && faabric::transport::isHostAlias(msg.executedhost())) {
        key += "@" + msg.executedhost();
    }
    return key;
}

static std::string executorKey(const faabric::Message& msg)
{
    return Scheduler::executorKeyFor(msg);
}

std::shared_ptr<faabric::executor::Executor> Scheduler::claimExecutor(
  faabric::Message& msg,
  std::unique_lock<std::shared_mutex>& schedulerLock)
{
    return claimExecutorForKey(executorKey(msg), msg, schedulerLock);
}

std::shared_ptr<faabric::executor::Executor> Scheduler::claimExecutorForKey(
  const std::string& key,
  faabric::Message& msg,
  std::unique_lock<std::shared_mutex>& schedulerLock)
{
    // Fast path: somebody told us they are idle
    for (;;) {
        std::shared_ptr<faabric::executor::Executor> candidate;
        {
            std::lock_guard<IdleLock> lk(idleMx);
            auto it = idleExecutors.find(key);
            if (it == idleExecutors.end() || it->second.empty()) {
                break;
            }
            candidate = it->second.back().lock();
            it->second.pop_back();
        }
        if (candidate != nullptr && !candidate->isShutdown() && candidate->tryClaim()) {
            SPDLOG_DEBUG("Reusing warm executor {} for {}", candidate->id, key);
            return candidate;
        }
    }
    auto& vec = executors[key];
    for (auto& e : vec) {
        if (e->tryClaim()) {
            SPDLOG_DEBUG("Reusing warm executor {} for {}", e->id, key);
            return e;
        }
    }
    // Creating an executor can be slow (memory set-up): do it unlocked
    SPDLOG_DEBUG("Scaling {} from {} -> {}", key, vec.size(), vec.size() + 1);
    schedulerLock.unlock();
    std::shared_ptr<faabric::executor::Executor> e;
    try {
        e = faabric::executor::getExecutorFactory()->createExecutor(msg);
    } catch (...) {
        schedulerLock.lock();
        throw;
    }
    schedulerLock.lock();
    e->claim();
    executors[key].push_back(e);
    return e;
}

// Starting a function costs a thread wake-up (a few microseconds of the
// caller's time each).  A wide batch is launched as a tree: half of what is left
// is handed to the pool thread woken next, which launches it before running its
// own message, so 128 functions are running after ~7 wake-up latencies instead
// of after 128 wake-ups issued by one thread.
namespace {
using LaunchList = std::vector<std::pair<std::shared_ptr<faabric::executor::Executor>, int>>;
constexpr int LAUNCH_TREE_LEAF = 4;

void launchTree(std::shared_ptr<LaunchList> list, int lo, int hi, std::shared_ptr<faabric::BatchExecuteRequest> req)
{
    if (hi < 0) {
        hi = (int)list->size();
    }
    while (hi - lo > LAUNCH_TREE_LEAF) {
        int mid = lo + (hi - lo) / 2;
        // [mid + 1, hi) travels with element `mid`
        int subLo = mid + 1, subHi = hi;
        std::function<void()> rest;
        if (subHi > subLo) {
            rest = [list, subLo, subHi, req] { launchTree(list, subLo, subHi, req); };
        }
        (*list)[mid].first->executeTasks({ (*list)[mid].second }, req, std::move(rest));
        hi = mid;
    }
    for (int i = lo; i < hi; i++) {
        (*list)[i].first->executeTasks({ (*list)[i].second }, req);
    }
}
}

void Scheduler::executeBatch(std::shared_ptr<faabric::BatchExecuteRequest> req)
{
    std::unique_lock<std::shared_mutex> lock(mx);
    bool isThreads = req->type() == faabric::BatchExecuteRequest::THREADS;
    int n = req->messages_size();
    if (n == 0) {
        return;
    }
    if (faabric::util::isTestMode()) {
        for (int i = 0; i < n; i++) {
            recordedMessages.push_back(req->messages(i));
        }
    }
    if (isThreads) {
        // All threads of a batch share one executor (and its memory).  On the
        // main host that is the executor already running the app's main
        // function; elsewhere a fresh one is claimed and restored from the
        // main thread's snapshot.
        faabric::Message& first = *req->mutable_messages(0);
        std::shared_ptr<faabric::executor::Executor> e;
        try {
            // (several per-GPU virtual hosts may share this scheduler: threads
            // addressed to a host other than the main one get an executor -
            // and a GPU - of their own)
            const bool onMainHost = first.mainhost().empty() || first.executedhost().empty() ||
                                    first.mainhost() == first.executedhost() ||
                                    !faabric::transport::isHostAlias(first.executedhost());
            if (onMainHost) {
                auto& candidates = executors[executorKey(first)];
                for (auto& c : candidates) {
                    if (c->isExecuting() && c->getCurrentAppId() == first.appid()) {
                        e = c;
                        break;
                    }
                }
            }
            if (e == nullptr) {
                e = claimExecutor(first, lock);
            }
        } catch (const std::exception& ex) {
            SPDLOG_ERROR("Failed to claim executor for {}: {}", faabric::util::funcToString(first, false), ex.what());
            lock.unlock();
            for (int i = 0; i < n; i++) {
                auto m = std::make_shared<faabric::Message>(req->messages(i));
                m->set_returnvalue(1);
                m->set_outputdata(std::string("Failed to claim executor: ") + ex.what());
                faabric::planner::getPlannerClient().setMessageResult(m);
            }
            return;
        }
        lock.unlock();
        std::vector<int> idxs(n);
        for (int i = 0; i < n; i++) {
            idxs[i] = i;
        }
        e->executeTasks(idxs, req);
        return;
    }
    // One executor per message
    std::vector<std::pair<std::shared_ptr<faabric::executor::Executor>, int>> launches;
    std::vector<int> failed;
    std::string failure;
    // (the messages of one per-host request nearly always share their key:
    // build it once, not 128 times under the scheduler's lock)
    launches.reserve(n);
    const faabric::Message* keyOf = nullptr;
    std::string key;
    for (int i = 0; i < n; i++) {
        faabric::Message& m = *req->mutable_messages(i);
        try {
            if (keyOf == nullptr || m.user() != keyOf->user() || m.function() != keyOf->function() ||
                m.executedhost() != keyOf->executedhost()) {
                key = executorKey(m);
                keyOf = &m;
            }
            launches.emplace_back(claimExecutorForKey(key, m, lock), i);
        } catch (const std::exception& ex) {
            failure = ex.what();
            failed.push_back(i);
        }
    }
    lock.unlock();
    launchTree(std::make_shared<LaunchList>(std::move(launches)), 0, -1, req);
    for (int idx : failed) {
        auto m = std::make_shared<faabric::Message>(req->messages(idx));
        m->set_returnvalue(1);
        m->set_outputdata("Failed to claim executor: " + failure);
        faabric::planner::getPlannerClient().setMessageResult(m);
    }
}

void Scheduler::broadcastSnapshotDelete(const faabric::Message& msg, const std::string& snapshotKey)
{
    for (const auto& host : faabric::planner::getPlannerClient().getAvailableHosts()) {
        if (host.ip() == thisHost || host.ip() == msg.mainhost()) {
            continue;
        }
        faabric::snapshot::getSnapshotClient(host.ip())->deleteSnapshot(snapshotKey);
    }
}

// ---------------------------------------------------------------------------
// Thread results
// ---------------------------------------------------------------------------
void Scheduler::setThreadResultLocally(uint32_t appId,
                                       uint32_t msgId,
                                       int32_t returnValue,
                                       faabric::transport::Message& message)
{
    // Diffs attached to the result point into the transport message: keep it
    // (a borrowed in-process view must first take a copy).  The result itself
    // reaches whoever awaits the thread through the planner, never from here:
    // the planner releases the thread's slot before it answers, so a function
    // that forks again right after the join finds its slots free
    // (reference: src/scheduler/Scheduler.cpp:395-421)
    std::lock_guard<std::mutex> lk(threadResultsMx);
    message.ensureOwned();
    threadResultMessages.insert_or_assign(msgId, std::move(message));
}

std::vector<std::pair<uint32_t, int32_t>> Scheduler::awaitThreadResults(
  std::shared_ptr<faabric::BatchExecuteRequest> req,
  int timeoutMs)
{
    std::vector<std::pair<uint32_t, int32_t>> results;
    results.reserve(req->messages_size());
    for (int i = 0; i < req->messages_size(); i++) {
        uint32_t msgId = (uint32_t)req->messages(i).id();
        faabric::Message res = faabric::planner::getPlannerClient().getMessageResult(
          req->appid(), (int)msgId, timeoutMs);
        if (res.type() == faabric::Message::EMPTY && res.id() != (int)msgId) {
            // Nothing came back in time: the join must not look like a success
            SPDLOG_ERROR("Timed out after {} ms waiting for thread {} of app {}", timeoutMs, msgId, req->appid());
            results.emplace_back(msgId, 1);
            continue;
        }
        results.emplace_back(msgId, res.returnvalue());
    }
    return results;
}

size_t Scheduler::getCachedMessageCount()
{
    std::lock_guard<std::mutex> lk(threadResultsMx);
    return threadResultMessages.size();
}

std::vector<faabric::Message> Scheduler::getRecordedMessages()
{
    std::shared_lock<std::shared_mutex> lock(mx);
    return recordedMessages;
}

void Scheduler::clearRecordedMessages()
{
    std::unique_lock<std::shared_mutex> lock(mx);
    recordedMessages.clear();
}

// ---------------------------------------------------------------------------
// Migration
// ---------------------------------------------------------------------------
std::shared_ptr<faabric::PendingMigration> Scheduler::checkForMigrationOpportunities(
  faabric::Message& msg,
  int overwriteNewGroupId)
{
    int appId = msg.appid();
    int groupId = msg.groupid();
    int groupIdx = msg.groupidx();
    SPDLOG_DEBUG("Message {}:{}:{} checking for migration opportunities", appId, groupId, groupIdx);

    int newGroupId = 0;
    if (groupIdx == 0) {
        // Idx 0 asks the planner on behalf of the group, then tells the rest
        auto req = std::make_shared<faabric::BatchExecuteRequest>();
        req->set_appid(appId);
        req->set_groupid(groupId);
        req->set_user(msg.user());
        req->set_function(msg.function());
        req->set_type(faabric::BatchExecuteRequest::MIGRATION);
        *req->add_messages() = msg;
        auto decision = faabric::planner::getPlannerClient().callFunctions(req);
        if ((int)decision.appId == DO_NOT_MIGRATE || (int)decision.appId == NOT_ENOUGH_SLOTS) {
            newGroupId = groupId;
        } else if ((int)decision.appId == MUST_FREEZE) {
            newGroupId = MUST_FREEZE;
        } else {
            newGroupId = decision.groupId;
        }
        if (overwriteNewGroupId != 0) {
            newGroupId = overwriteNewGroupId;
        }
        std::vector<uint8_t> bytes(sizeof(int));
        memcpy(bytes.data(), &newGroupId, sizeof(int));
        auto idxs = broker.getIdxsRegisteredForGroup(groupId);
        for (int idx : idxs) {
            if (idx != 0) {
                broker.sendMessage(groupId, 0, idx, bytes.data(), bytes.size());
            }
        }
    } else if (overwriteNewGroupId == 0) {
        std::vector<uint8_t> bytes = broker.recvMessage(groupId, 0, groupIdx);
        memcpy(&newGroupId, bytes.data(), sizeof(int));
    } else {
        newGroupId = overwriteNewGroupId;
    }

    if (newGroupId == MUST_FREEZE) {
        // Signalled through a pending migration to "nowhere"
        auto frozen = std::make_shared<faabric::PendingMigration>();
        frozen->set_appid(MUST_FREEZE);
        return frozen;
    }
    if (newGroupId == groupId) {
        return nullptr; // nothing to do
    }
    // The planner pushed the new mappings before answering idx 0
    msg.set_groupid(newGroupId);
    broker.waitForMappingsOnThisHost(newGroupId);
    std::string newHost = broker.getHostForReceiver(newGroupId, groupIdx);
    auto migration = std::make_shared<faabric::PendingMigration>();
    migration->set_appid(appId);
    migration->set_groupid(newGroupId);
    migration->set_groupidx(groupIdx);
    migration->set_srchost(msg.executedhost().empty() ? thisHost : msg.executedhost());
    migration->set_dsthost(newHost);
    return migration;
}

} // namespace faabric::scheduler
