// GpuPPOAgent.cs -- the reference's PPOAgent surface (Walker/PPO/PPOAgent.cs:23 ctor, :147 Train(Trajectory, Renderer),
// :192 Save, :381 SampleActions) forwarding to libwalker_b200's wb_policy_* exports.  Source only (no .NET toolchain in the
// build image); see INTEGRATION.md.  Host-side pieces the reference keeps in C# stay in C# here: the network DSL
// (ParseLayers), Xavier initialisation (Matrix.FromXavier), the System.Random draws of the Box-Muller transform, the
// shuffling of CreateBatches and the .weights text format.  Forward passes, the clipped-surrogate gradient, the backward
// pass, Adam and the return / advantage recurrences run in the library.
using System;
using System.Collections.Generic;
using System.IO;
using System.Linq;
using System.Text.RegularExpressions;
using NEA.Native;
using NEA.Rendering;
using NEA.Walker.PPO.Network;

namespace NEA.Walker.PPO;

public sealed class GpuPPOAgent : IDisposable
{
    private readonly IntPtr _policy;
    private readonly int _stateSize, _actionSize;
    private readonly List<(int outSize, int inSize)> _actorDense = new(), _criticDense = new();
    private readonly Random _random = new Random();
    private const string WeightsLocation = "Data/Weights/";     // PPOAgent.cs:21

    // new PPOAgent(stateSize, actionSize) (PPOAgent.cs:23-37): parse both DSL strings (falling back to the defaults like
    // CreateNetworks, :41-93), create the device networks, Xavier-initialise, then Load("critic") / Load("actor").
    public GpuPPOAgent(int stateSize, int actionSize)
    {
        _stateSize = stateSize;
        _actionSize = actionSize;
        ParseNetworks(actionSize, out var ak, out var asz, out var ck, out var cs);
        var hp = WbHyperparams.FromStatics();
        Wb.Ok(Wb.wb_init(0), "wb_init");
        Wb.Ok(Wb.wb_policy_create(stateSize, actionSize, ak, asz, ak.Length, ck, cs, ck.Length, ref hp, out _policy), "wb_policy_create");
        DenseShapes(stateSize, ak, asz, _actorDense);
        DenseShapes(stateSize, ck, cs, _criticDense);
        Wb.Ok(Wb.wb_policy_set_weights(_policy, 1, Xavier(_criticDense)), "wb_policy_set_weights(critic)");
        Wb.Ok(Wb.wb_policy_set_weights(_policy, 0, Xavier(_actorDense)), "wb_policy_set_weights(actor)");
        Load("critic");
        Load("actor");
    }

    internal IntPtr Handle => _policy;

    // PPOAgent.CreateNetworks (PPOAgent.cs:41-93): parse Hyperparameters.CriticNeuralNetwork / ActorNeuralNetwork; a string that does
    // not parse, or whose last dense layer is not 1 / actionSize wide, is logged and replaced by the default network
    internal static void ParseNetworks(int actionSize, out int[] ak, out int[] asz, out int[] ck, out int[] cs)
    {
        const string defaultCritic = "Input |64| (LeakyReLU) |1| Output", defaultActor = "Input |64| (LeakyReLU) |64| (LeakyReLU) |4| (TanH) Output";
        if (!TryParse(Hyperparameters.CriticNeuralNetwork, out ck, out cs) || cs.Last(s => s > 0) != 1)
        {
            ErrorLogger.LogError("Exception occurred while attempting to parse the critic neural network.");
            Hyperparameters.CriticNeuralNetwork = defaultCritic;
            TryParse(defaultCritic, out ck, out cs);
        }
        if (!TryParse(Hyperparameters.ActorNeuralNetwork, out ak, out asz) || asz.Last(s => s > 0) != actionSize)
        {
            ErrorLogger.LogError("Exception occurred while attempting to parse the actor neural network.");
            Hyperparameters.ActorNeuralNetwork = defaultActor;
            TryParse(defaultActor, out ak, out asz);
        }
    }

    // PPOAgent.ParseLayers (PPOAgent.cs:96-143) -> kinds / sizes for wb_policy_create
    private static bool TryParse(string structure, out int[] kinds, out int[] sizes)
    {
        kinds = sizes = Array.Empty<int>();
        if (!Regex.IsMatch(structure, @"^Input( \|\d+\|| \((ReLU|TanH|LeakyReLU)\))+ Output$")) return false;
        string cleaned = Regex.Replace(structure, @"[\[|()]|( Output)|(Input )", "");
        var k = new List<int>();
        var s = new List<int>();
        foreach (var token in cleaned.Split(' '))
        {
            if (int.TryParse(token, out int size)) { k.Add(Wb.Dense); s.Add(size); }
            else { k.Add(token == "ReLU" ? Wb.ReLU : token == "LeakyReLU" ? Wb.LeakyReLU : Wb.TanH); s.Add(0); }
        }
        kinds = k.ToArray();
        sizes = s.ToArray();
        return k.Contains(Wb.Dense);
    }

    internal static void DenseShapes(int input, int[] kinds, int[] sizes, List<(int, int)> shapes)
    {
        int width = input;
        for (int i = 0; i < kinds.Length; i++)
            if (kinds[i] == Wb.Dense) { shapes.Add((sizes[i], width)); width = sizes[i]; }
    }

    // DenseLayer ctor (DenseLayer.cs:22-33): weights Matrix.FromXavier(out, in) (Matrix.cs:59-80), zero biases;
    // flat layout per dense layer W[out][in] row-major then b[out] (DenseLayer.Save order)
    internal static float[] Xavier(List<(int outSize, int inSize)> shapes)
    {
        var flat = new List<float>();
        foreach (var (o, i) in shapes)
        {
            flat.AddRange(Matrix.GetRepresentation(Matrix.FromXavier(o, i)));
            flat.AddRange(new float[o]);
        }
        return flat.ToArray();
    }

    // PPOAgent.SampleActions (PPOAgent.cs:381-398) for one state: the mean comes from the device actor, the two uniforms of
    // every Box-Muller draw from System.Random like Matrix.SampleNormal (Matrix.cs:541-555, NormalDistribution.cs:12-20)
    public Matrix SampleActions(Matrix state, out Matrix logProbabilities, out Matrix mean, out Matrix std)
    {
        var actions = new float[_actionSize];
        var logp = new float[_actionSize];
        var mu = new float[_actionSize];
        SampleActions(1, Matrix.GetRepresentation(state), actions, logp, mu);
        logProbabilities = Matrix.FromValues(logp);
        mean = Matrix.FromValues(mu);
        std = Matrix.FromValues(Enumerable.Repeat(MathF.Exp(Hyperparameters.LogStandardDeviation), _actionSize).ToArray());   // GetStandardDeviations, :367-378
        return Matrix.FromValues(actions);
    }

    // the same for n walkers at once: states [n][stateSize] -> actions / logp / mean [n][actionSize]
    public void SampleActions(int n, float[] states, float[] actions, float[] logp, float[] mean)
    {
        var uniforms = new float[n * _actionSize * 2];
        for (int i = 0; i < uniforms.Length; i++) uniforms[i] = (float)_random.NextDouble();
        Wb.Ok(Wb.wb_policy_sample(_policy, n, states, uniforms, actions, logp, mean), "wb_policy_sample");
    }

    // PPOAgent.GetValueEstimate (PPOAgent.cs:350-364) for n states
    public float[] ValueEstimates(int n, float[] states)
    {
        var values = new float[n];
        Wb.Ok(Wb.wb_policy_forward(_policy, n, states, null, values), "wb_policy_forward");
        return values;
    }

    // PPOAgent.Train(Trajectory, Renderer) (PPOAgent.cs:147-172)
    public void Train(Trajectory trajectory, Renderer renderer)
    {
        int T = trajectory.States.Count;
        if (T == 0) return;
        var hp = WbHyperparams.FromStatics();                      // the static hyper-parameters may have been edited in the menu
        Wb.Ok(Wb.wb_policy_set_hyperparams(_policy, ref hp), "wb_policy_set_hyperparams");
        float[] states = Flatten(trajectory.States, _stateSize), actions = Flatten(trajectory.Actions, _actionSize);
        float[] logp = Flatten(trajectory.LogProbabilities, _actionSize), rewards = trajectory.Rewards.ToArray();
        // CalculateValues (:175-189): value estimates, MC return / GAE, optional Normalize
        float[] values = ValueEstimates(T, states), returns = new float[T], advantages = new float[T];
        Wb.Ok(Wb.wb_returns_advantages(_policy, T, rewards, values, returns, advantages), "wb_returns_advantages");
        trajectory.Values.Clear(); trajectory.Values.AddRange(values);
        trajectory.Returns.Clear(); trajectory.Returns.AddRange(returns);
        trajectory.Advantages.Clear(); trajectory.Advantages.AddRange(advantages);
        renderer.AddTotalEpisodeReward(trajectory.Rewards.Sum());

        int B = Hyperparameters.BatchSize, batchCount = T / B;
        var losses = new float[2];
        float[] bs = new float[B * _stateSize], ba = new float[B * _actionSize], bl = new float[B * _actionSize], badv = new float[B], bret = new float[B];
        for (int epoch = 0; epoch < Hyperparameters.Epochs; epoch++)
        {
            // CreateBatches (:501-540): sampling without replacement, the remainder is dropped
            var pool = Enumerable.Range(0, T).ToList();
            for (int j = 0; j < batchCount; j++)
            {
                for (int b = 0; b < B; b++)
                {
                    int pick = _random.Next(0, pool.Count), idx = pool[pick];
                    pool.RemoveAt(pick);
                    Array.Copy(states, idx * _stateSize, bs, b * _stateSize, _stateSize);
                    Array.Copy(actions, idx * _actionSize, ba, b * _actionSize, _actionSize);
                    Array.Copy(logp, idx * _actionSize, bl, b * _actionSize, _actionSize);
                    badv[b] = advantages[idx];
                    bret[b] = returns[idx];
                }
                // Train(Batch) (:218-346): Zero, per-sample clipped-surrogate + value gradients, FeedBack, Optimise -- one call,
                // one kernel launch on the default networks (wb_ppo_grad + wb_adam_step are the two halves)
                Wb.Ok(Wb.wb_ppo_train(_policy, B, bs, ba, bl, badv, bret, losses, out _), "wb_ppo_train");
                renderer.UpdateConsole(epoch, j, batchCount, losses[0]);
            }
        }
        renderer.AddCriticLoss(losses[0]);
        renderer.AddActorLoss(losses[1]);
        if (Hyperparameters.SaveWeights) Save();
    }

    // Train(Trajectory, Renderer) for every finished episode of the list, in list order, as ONE native call
    // (wb_ppo_train_trajectories: one kernel launch on the default networks).  CreateBatches is drawn from _random in the order
    // the single-trajectory overload draws it, so the mini-batches are the same.  Deviation: the per-mini-batch
    // renderer.UpdateConsole becomes one update per trajectory (its last mini-batch), since the mini-batches run on the device.
    public void Train(IReadOnlyList<Trajectory> trajectories, Renderer renderer)
    {
        var hp = WbHyperparams.FromStatics();
        Wb.Ok(Wb.wb_policy_set_hyperparams(_policy, ref hp), "wb_policy_set_hyperparams");
        int n = trajectories.Count, B = Hyperparameters.BatchSize, epochs = Hyperparameters.Epochs;
        if (n == 0) return;
        var offsets = new int[n + 1];
        for (int e = 0; e < n; e++) offsets[e + 1] = offsets[e] + trajectories[e].States.Count;
        int rows = offsets[n];
        float[] states = new float[rows * _stateSize], actions = new float[rows * _actionSize], logp = new float[rows * _actionSize];
        float[] rewards = new float[rows];
        var index = new List<int>();
        for (int e = 0; e < n; e++)
        {
            var t = trajectories[e];
            int T = t.States.Count, o = offsets[e];
            Array.Copy(Flatten(t.States, _stateSize), 0, states, o * _stateSize, T * _stateSize);
            Array.Copy(Flatten(t.Actions, _actionSize), 0, actions, o * _actionSize, T * _actionSize);
            Array.Copy(Flatten(t.LogProbabilities, _actionSize), 0, logp, o * _actionSize, T * _actionSize);
            t.Rewards.CopyTo(rewards, o);
            for (int epoch = 0; epoch < epochs; epoch++)  // CreateBatches (:501-540), as in Train(Trajectory, Renderer)
            {
                var pool = Enumerable.Range(0, T).ToList();
                for (int j = 0; j < T / B; j++)
                    for (int b = 0; b < B; b++)
                    {
                        int pick = _random.Next(0, pool.Count);
                        index.Add(pool[pick]);
                        pool.RemoveAt(pick);
                    }
            }
        }
        float[] values = new float[rows], returns = new float[rows], advantages = new float[rows], losses = new float[2 * n];
        var skipped = new int[n];
        Wb.Ok(Wb.wb_ppo_train_trajectories(_policy, n, offsets, epochs, states, actions, logp, rewards, index.ToArray(), values, returns,
                                           advantages, losses, skipped), "wb_ppo_train_trajectories");
        for (int e = 0; e < n; e++)
        {
            var t = trajectories[e];
            int T = t.States.Count, o = offsets[e];
            if (T == 0) continue;  // Train returns before anything is recorded
            t.Values.Clear(); t.Values.AddRange(new ArraySegment<float>(values, o, T));
            t.Returns.Clear(); t.Returns.AddRange(new ArraySegment<float>(returns, o, T));
            t.Advantages.Clear(); t.Advantages.AddRange(new ArraySegment<float>(advantages, o, T));
            renderer.AddTotalEpisodeReward(t.Rewards.Sum());
            if (T >= B) renderer.UpdateConsole(epochs - 1, T / B - 1, T / B, losses[2 * e]);
            renderer.AddCriticLoss(losses[2 * e]);
            renderer.AddActorLoss(losses[2 * e + 1]);
        }
        if (Hyperparameters.SaveWeights) Save();
    }

    internal static float[] Flatten(List<Matrix> rows, int width)
    {
        var flat = new float[rows.Count * width];
        for (int t = 0; t < rows.Count; t++)
            for (int k = 0; k < width; k++) flat[t * width + k] = rows[t].GetValue(k, 0);
        return flat;
    }

    // NeuralNetwork.Save (NeuralNetwork.cs:159-176) + PPOAgent.Save (PPOAgent.cs:192-213): structure line, then per dense layer
    // "W <weights> B <biases>" (DenseLayer.Save, DenseLayer.cs:73-79)
    public void Save()
    {
        Hyperparameters.CreateDirectories();
        File.WriteAllLines($"{Hyperparameters.FilePath}{WeightsLocation}{Hyperparameters.CriticWeightFileName}.weights", Lines(1, Hyperparameters.CriticNeuralNetwork, _criticDense));
        File.WriteAllLines($"{Hyperparameters.FilePath}{WeightsLocation}{Hyperparameters.ActorWeightFileName}.weights", Lines(0, Hyperparameters.ActorNeuralNetwork, _actorDense));
    }

    private string[] Lines(int which, string structure, List<(int outSize, int inSize)> shapes)
    {
        Wb.wb_policy_num_params(_policy, which, out int count);
        var flat = new float[count];
        Wb.Ok(Wb.wb_policy_get_weights(_policy, which, flat), "wb_policy_get_weights");
        var lines = new List<string> { structure };
        int p = 0;
        foreach (var (o, i) in shapes)
        {
            string w = string.Join(" ", flat.Skip(p).Take(o * i));
            p += o * i;
            string b = string.Join(" ", flat.Skip(p).Take(o));
            p += o;
            lines.Add("W " + w + " B " + b);
        }
        return lines.ToArray();
    }

    // NeuralNetwork.Load (NeuralNetwork.cs:94-115): structure line must match, ValidateWeights on every line, then the lines that
    // are present replace the leading dense layers
    public void Load(string type)
    {
        int which = type == "critic" ? 1 : 0;
        Wb.wb_policy_num_params(_policy, which, out int count);
        var flat = new float[count];
        Wb.Ok(Wb.wb_policy_get_weights(_policy, which, flat), "wb_policy_get_weights");
        if (LoadInto(type, type == "critic" ? _criticDense : _actorDense, flat))
            Wb.Ok(Wb.wb_policy_set_weights(_policy, which, flat), "wb_policy_set_weights");
    }

    // the weights file of `type` (Hyperparameters.CriticWeights / ActorWeights) over one network's flat parameters; false: nothing loaded
    internal static bool LoadInto(string type, List<(int outSize, int inSize)> shapes, float[] flat)
    {
        string[] contents = type == "critic" ? Hyperparameters.CriticWeights : Hyperparameters.ActorWeights;
        string network = type == "critic" ? Hyperparameters.CriticNeuralNetwork : Hyperparameters.ActorNeuralNetwork;
        if (contents.Length < 2 || contents[0] != network) return false;
        (bool ok, _) = NeuralNetwork.ValidateWeights(contents);
        if (!ok || contents.Length - 1 > shapes.Count) return false;
        var loaded = (float[])flat.Clone();
        int p = 0;
        for (int l = 0; l < contents.Length - 1; l++)
        {
            var (o, i) = shapes[l];
            string line = contents[l + 1];
            int wi = line.IndexOf("W", StringComparison.Ordinal) + 2, bi = line.IndexOf("B", StringComparison.Ordinal) + 2;
            float[] w = Array.ConvertAll(line.Substring(wi, bi - wi - 3).Split(), float.Parse);
            float[] b = Array.ConvertAll(line.Substring(bi).Split(), float.Parse);
            if (w.Length < o * i || b.Length < o) return false;     // Matrix.Load would throw (Matrix.cs:118-127)
            Array.Copy(w, 0, loaded, p, o * i);
            p += o * i;
            Array.Copy(b, 0, loaded, p, o);
            p += o;
        }
        loaded.CopyTo(flat, 0);
        return true;
    }

    public void Dispose() => Wb.wb_policy_destroy(_policy);
}

// One PPO brain per walker: P agents with the networks of Hyperparameters.ActorNeuralNetwork / CriticNeuralNetwork (parsed, with
// the reference's fallbacks, as GpuPPOAgent parses them) on one native handle (wb_population_*).  In the reference every walker owns its PPOAgent (Walker.cs:25-34) and trains it on each of its own episodes
// (Environment.cs:91,157-164); agent a here is one GpuPPOAgent with its own weights, Adam state and step counters.  The
// hyper-parameters are the statics at construction.  Xavier initialisation, the Box-Muller uniforms and CreateBatches are drawn
// from System.Random in C#, as GpuPPOAgent draws them.
public sealed class GpuPopulation : IDisposable
{
    private readonly IntPtr _population;
    private readonly int _n;
    private readonly Random _random = new Random();
    private readonly List<(int outSize, int inSize)> _actorDense = new(), _criticDense = new();

    // new PPOAgent(12, 4) per agent (PPOAgent.cs:23-37): the networks of the DSL strings, Xavier initialisation (critic first, then
    // actor), then Load("critic") / Load("actor") when weights are set
    public GpuPopulation(int agents)
    {
        _n = agents;
        GpuPPOAgent.ParseNetworks(Wb.Act, out var ak, out var asz, out var ck, out var cs);
        var hp = Enumerable.Repeat(WbHyperparams.FromStatics(), agents).ToArray();
        Wb.Ok(Wb.wb_init(0), "wb_init");
        Wb.Ok(Wb.wb_population_create_net(agents, Wb.Obs, Wb.Act, ak, asz, ak.Length, ck, cs, ck.Length, ref hp[0], out _population),
              "wb_population_create_net");
        GpuPPOAgent.DenseShapes(Wb.Obs, ak, asz, _actorDense);
        GpuPPOAgent.DenseShapes(Wb.Obs, ck, cs, _criticDense);
        for (int a = 0; a < agents; a++)
        {
            float[] critic = GpuPPOAgent.Xavier(_criticDense), actor = GpuPPOAgent.Xavier(_actorDense);
            GpuPPOAgent.LoadInto("critic", _criticDense, critic);
            GpuPPOAgent.LoadInto("actor", _actorDense, actor);
            Wb.Ok(Wb.wb_population_set_weights(_population, a, actor.Concat(critic).ToArray()), "wb_population_set_weights");
        }
    }

    public int Count => _n;

    // PPOAgent.SampleActions (PPOAgent.cs:381-398) of every agent on its walker's state: states [n][12] -> actions / logp / mean [n][4]
    public void SampleActions(int n, float[] states, float[] actions, float[] logp, float[] mean)
    {
        var uniforms = new float[n * Wb.Act * 2];
        for (int i = 0; i < uniforms.Length; i++) uniforms[i] = (float)_random.NextDouble();
        Wb.Ok(Wb.wb_population_sample(_population, n, states, uniforms, actions, logp, mean), "wb_population_sample");
    }

    // one agent's action on `state`, the other walkers' states as given (the native call samples every agent)
    public Matrix SampleAction(int agent, float[] state, float[] states, out Matrix logProbabilities)
    {
        var all = (float[])states.Clone();
        Array.Copy(state, 0, all, agent * Wb.Obs, Wb.Obs);
        float[] actions = new float[_n * Wb.Act], logp = new float[_n * Wb.Act], mean = new float[_n * Wb.Act];
        SampleActions(_n, all, actions, logp, mean);
        logProbabilities = Matrix.FromValues(logp.Skip(agent * Wb.Act).Take(Wb.Act).ToArray());
        return Matrix.FromValues(actions.Skip(agent * Wb.Act).Take(Wb.Act).ToArray());
    }

    // PPOAgent.Train(Trajectory, Renderer) (PPOAgent.cs:147-172) of each listed agent on its episodes, in list order, as ONE native
    // call (wb_population_train_trajectories: one kernel launch).  CreateBatches is drawn in list order, as calling
    // GpuPPOAgent.Train per episode would draw it; the console is updated once per episode, as in GpuPPOAgent's list overload.
    public void Train(IReadOnlyList<(int agent, Trajectory trajectory)> episodes, Renderer renderer)
    {
        int n = episodes.Count, B = Hyperparameters.BatchSize, epochs = Hyperparameters.Epochs;
        if (n == 0) return;
        var agents = new int[n];
        var offsets = new int[n + 1];
        for (int e = 0; e < n; e++) { agents[e] = episodes[e].agent; offsets[e + 1] = offsets[e] + episodes[e].trajectory.States.Count; }
        int rows = offsets[n];
        float[] states = new float[rows * Wb.Obs], actions = new float[rows * Wb.Act], logp = new float[rows * Wb.Act], rewards = new float[rows];
        var index = new List<int>();
        for (int e = 0; e < n; e++)
        {
            var t = episodes[e].trajectory;
            int T = t.States.Count, o = offsets[e];
            Array.Copy(GpuPPOAgent.Flatten(t.States, Wb.Obs), 0, states, o * Wb.Obs, T * Wb.Obs);
            Array.Copy(GpuPPOAgent.Flatten(t.Actions, Wb.Act), 0, actions, o * Wb.Act, T * Wb.Act);
            Array.Copy(GpuPPOAgent.Flatten(t.LogProbabilities, Wb.Act), 0, logp, o * Wb.Act, T * Wb.Act);
            t.Rewards.CopyTo(rewards, o);
            for (int epoch = 0; epoch < epochs; epoch++)  // CreateBatches (:501-540): sampling without replacement
            {
                var pool = Enumerable.Range(0, T).ToList();
                for (int j = 0; j < T / B; j++)
                    for (int b = 0; b < B; b++)
                    {
                        int pick = _random.Next(0, pool.Count);
                        index.Add(pool[pick]);
                        pool.RemoveAt(pick);
                    }
            }
        }
        float[] values = new float[rows], returns = new float[rows], advantages = new float[rows], losses = new float[2 * n];
        var skipped = new int[n];
        Wb.Ok(Wb.wb_population_train_trajectories(_population, n, agents, offsets, epochs, states, actions, logp, rewards, index.ToArray(),
                                                   values, returns, advantages, losses, skipped), "wb_population_train_trajectories");
        for (int e = 0; e < n; e++)
        {
            var t = episodes[e].trajectory;
            int T = t.States.Count, o = offsets[e];
            if (T == 0) continue;
            t.Values.Clear(); t.Values.AddRange(new ArraySegment<float>(values, o, T));
            t.Returns.Clear(); t.Returns.AddRange(new ArraySegment<float>(returns, o, T));
            t.Advantages.Clear(); t.Advantages.AddRange(new ArraySegment<float>(advantages, o, T));
            renderer.AddTotalEpisodeReward(t.Rewards.Sum());
            if (T >= B) renderer.UpdateConsole(epochs - 1, T / B - 1, T / B, losses[2 * e]);
            renderer.AddCriticLoss(losses[2 * e]);
            renderer.AddActorLoss(losses[2 * e + 1]);
        }
    }

    public void Dispose() => Wb.wb_population_destroy(_population);
}
