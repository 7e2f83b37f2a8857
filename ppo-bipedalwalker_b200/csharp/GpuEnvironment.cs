// GpuEnvironment.cs -- the reference's Environment surface (Environment.cs:56 GetConsoleInformation, :64 Update(float),
// :126 StepObjects(float), :176 InitialState) for N lockstep walkers on libwalker_b200.  Source only (no .NET toolchain in
// the build image); see INTEGRATION.md.
//
// Update(deltaTime) keeps the reference's signature and loop -- observe state, sample action, TakeActions(Clip), step physics,
// receive reward, train on terminal -- for ALL walkers per call: one wb_policy_sample, one fused wb_env_step (which also resets
// the walkers that terminated and returns their initial observation, Environment.cs:167-180), N trajectories, and
// PPOAgent.Train on the trajectory of every walker whose episode just ended (one shared brain, like N copies of the
// reference training the same weights files).  With brainPerWalker every walker owns its agent, as in the reference (Walker.cs:25-34):
// the actions come from one wb_population_sample and every walker whose episode ended in the step trains its own agent, all in
// one wb_population_train_trajectories call.
using System;
using System.Collections.Generic;
using System.Linq;
using System.Runtime.InteropServices;
using Microsoft.Xna.Framework;
using NEA.Native;
using NEA.Rendering;
using NEA.Walker;
using NEA.Walker.PPO;
using Matrix = NEA.Walker.PPO.Matrix;

namespace NEA;

public class GpuEnvironment : IDisposable
{
    private readonly IntPtr _env;
    private readonly int _n;
    private readonly Renderer _renderer;
    private readonly GpuPPOAgent _brain;          // one shared brain (brainPerWalker: null)
    private readonly GpuPopulation _population;   // brainPerWalker: agent i is walker i's brain (otherwise null)
    private readonly GpuWalker[] _walkers;
    private readonly Trajectory[] _trajectories;
    private readonly int[] _steps;
    private readonly float[] _obs, _reward, _actions, _logp, _mean;
    private readonly byte[] _done;
    // the four I/O arrays stay pinned (GCHandle) and page-locked (wb_host_pin) for the life of the object: wb_env_step then
    // reads the actions and writes obs / reward / done through their device aliases (zero-copy path, include/walker_b200.h)
    private GCHandle _hObs, _hReward, _hActions, _hDone;
    // lazily fetched copy of the state records (renderer / joint queries): [92][N] floats, [2][N] ints
    private float[] _stateF;
    private int[] _stateI;
    private bool _stateFresh;
    private readonly Vector2[] _position, _previousPosition;
    private int _episodes;
    private float _bestDistance, _previousAverageReward;

    public GpuEnvironment(Renderer renderer, int walkers = 1, Wb.Material floorMaterial = Wb.Material.Metal /* Environment.cs:223 */,
                          bool brainPerWalker = false)
    {
        _n = walkers;
        _renderer = renderer;
        var hp = WbHyperparams.FromStatics();
        var floors = Enumerable.Repeat((byte)floorMaterial, walkers).ToArray();
        Wb.Ok(Wb.wb_init(0), "wb_init");
        Wb.Ok(Wb.wb_env_create(walkers, floors, null, ref hp, out _env), "wb_env_create");
        if (brainPerWalker) _population = new GpuPopulation(walkers);
        else _brain = new GpuPPOAgent(Wb.Obs, Wb.Act);
        _walkers = Enumerable.Range(0, walkers).Select(i => new GpuWalker(this, i, _brain, _population)).ToArray();
        _trajectories = Enumerable.Range(0, walkers).Select(_ => new Trajectory()).ToArray();
        _steps = new int[walkers];
        _obs = new float[walkers * Wb.Obs];
        _reward = new float[walkers];
        _done = new byte[walkers];
        _actions = new float[walkers * Wb.Act];
        _logp = new float[walkers * Wb.Act];
        _mean = new float[walkers * Wb.Act];
        _stateF = new float[Wb.StateFloats * walkers];
        _stateI = new int[Wb.StateInts * walkers];
        _position = Enumerable.Repeat(new Vector2(125, 800), walkers).ToArray();      // Walker.cs:31
        _previousPosition = (Vector2[])_position.Clone();
        _hObs = Pin(_obs, sizeof(float) * _obs.Length);
        _hReward = Pin(_reward, sizeof(float) * _reward.Length);
        _hActions = Pin(_actions, sizeof(float) * _actions.Length);
        _hDone = Pin(_done, _done.Length);
        InitialState();
    }

    public int Count => _n;
    public GpuWalker Walker(int index) => _walkers[index];

    private static GCHandle Pin(Array a, int bytes)
    {
        var h = GCHandle.Alloc(a, GCHandleType.Pinned);
        Wb.Ok(Wb.wb_host_pin(h.AddrOfPinnedObject(), (UIntPtr)bytes), "wb_host_pin");
        return h;
    }

    private static void Unpin(ref GCHandle h)
    {
        if (!h.IsAllocated) return;
        Wb.wb_host_unpin(h.AddrOfPinnedObject());
        h.Free();
    }

    // Environment.GetConsoleInformation (Environment.cs:56-60) for walker 0 (the one the console renderer follows)
    public (int, int, float, float, float, float, Matrix) GetConsoleInformation()
    {
        var rewards = _trajectories[0].Rewards;
        float averageReward = rewards.Count == 0 ? 0 : rewards.Average();
        return (_episodes, _steps[0], _position[0].X, averageReward, _bestDistance, _previousAverageReward, _walkers[0].GetState());
    }

    // Environment.InitialState (Environment.cs:176-180): Walker.Update + GetState for every walker
    public void InitialState()
    {
        Wb.Ok(Wb.wb_env_get_obs(_env, _obs), "wb_env_get_obs");
        _stateFresh = false;
    }

    // Environment.StepObjects (Environment.cs:126-143) for every walker (deltaTime is divided by Hyperparameters.Iterations inside)
    public void StepObjects(float deltaTime)
    {
        Wb.Ok(Wb.wb_env_step_objects(_env, deltaTime), "wb_env_step_objects");
        _stateFresh = false;
    }

    // Environment.Update (Environment.cs:64-92), same signature, all N walkers
    public void Update(float deltaTime)
    {
        if (Console.KeyAvailable && Console.ReadKey(true).Key == ConsoleKey.X) _renderer.ExitTraining();
        for (int i = 0; i < _n; i++)
        {
            _trajectories[i].Indexes.Add(_steps[i]);
            _steps[i]++;
            _trajectories[i].States.Add(_walkers[i].GetState());
        }
        // _walker.GetActions(_state, out logProbabilities) for every walker: one batched forward + Box-Muller
        if (_population != null) _population.SampleActions(_n, _obs, _actions, _logp, _mean);
        else _brain.SampleActions(_n, _obs, _actions, _logp, _mean);
        var sampled = (float[])_actions.Clone();     // the trajectory stores the UNCLIPPED action (Environment.cs:87)
        // TakeActions(Matrix.Clip(action, 1, -1)) + Step + (on terminal) Reset + InitialState: one fused launch, zero-copy I/O
        Wb.Ok(Wb.wb_env_step_pinned(_env, _hActions.AddrOfPinnedObject(), deltaTime, 1, _hObs.AddrOfPinnedObject(),
                                    _hReward.AddrOfPinnedObject(), _hDone.AddrOfPinnedObject()), "wb_env_step");
        _stateFresh = false;
        var finished = new List<(int agent, Trajectory trajectory)>();
        for (int i = 0; i < _n; i++)
        {
            _trajectories[i].Actions.Add(Matrix.FromValues(sampled.Skip(i * Wb.Act).Take(Wb.Act).ToArray()));
            _trajectories[i].LogProbabilities.Add(Matrix.FromValues(_logp.Skip(i * Wb.Act).Take(Wb.Act).ToArray()));
            _trajectories[i].Rewards.Add(_reward[i]);
            _previousPosition[i] = _position[i];
            if (_done[i] == 0) continue;
            if (_population == null) TrainNetworks(i);
            else { finished.Add((i, _trajectories[i])); EndEpisode(i); }
        }
        // brainPerWalker: every walker whose episode ended trains its own agent, all in one native call
        if (finished.Count > 0) _population.Train(finished, _renderer);
        RefreshPositions();
    }

    // Environment.TrainNetworks + Reset (Environment.cs:157-173); the physical reset already happened inside the fused step
    private void TrainNetworks(int i)
    {
        _walkers[i].Train(_trajectories[i], _renderer);
        EndEpisode(i);
    }

    private void EndEpisode(int i)
    {
        _episodes++;
        if (i == 0) _previousAverageReward = _trajectories[i].Rewards.Average();
        _trajectories[i] = new Trajectory();
        _steps[i] = 0;
    }

    private void RefreshPositions()
    {
        FetchState();
        for (int i = 0; i < _n; i++)
        {
            // Body centroid: floats 58 + 2 * 2, 58 + 2 * 2 + 1 of the record (SoA: [float][walker])
            _position[i] = new Vector2(_stateF[62 * _n + i], _stateF[63 * _n + i]);
            if (_position[i].X > _bestDistance) _bestDistance = _position[i].X;
            if (_done[i] != 0) _previousPosition[i] = _position[i];       // Walker.Reset: _previousPosition = _position (Walker.cs:219-220)
        }
    }

    private void FetchState()
    {
        if (_stateFresh) return;
        Wb.Ok(Wb.wb_env_get_state(_env, _stateF, _stateI), "wb_env_get_state");
        _stateFresh = true;
    }

    // ---- what GpuWalker reads
    internal void StageAction(int walker, int joint, float torque)
    {
        _actions[walker * Wb.Act + joint] = torque;
        if (walker == _n - 1 && joint == Wb.Act - 1) { Wb.Ok(Wb.wb_env_take_actions(_env, _actions), "wb_env_take_actions"); _stateFresh = false; }
    }
    internal float[] Observation(int walker) => _obs.Skip(walker * Wb.Obs).Take(Wb.Obs).ToArray();
    internal float[] Observations() => (float[])_obs.Clone();
    internal Vector2 Position(int walker) => _position[walker];
    internal Vector2 PreviousPosition(int walker) => _previousPosition[walker];
    internal int Flags(int walker) { FetchState(); return _stateI[walker]; }
    internal float[] Record(int walker)
    {
        FetchState();
        var r = new float[Wb.StateFloats];
        for (int f = 0; f < Wb.StateFloats; f++) r[f] = _stateF[f * _n + walker];
        return r;
    }
    internal void ResetWalker(int walker)
    {
        var mask = new byte[_n];
        mask[walker] = 1;
        Wb.Ok(Wb.wb_env_reset(_env, mask, 0), "wb_env_reset");
        _stateFresh = false;
        InitialState();
    }

    public void Dispose()
    {
        Unpin(ref _hObs);
        Unpin(ref _hReward);
        Unpin(ref _hActions);
        Unpin(ref _hDone);
        Wb.wb_env_destroy(_env);
        _brain?.Dispose();
        _population?.Dispose();
    }
}
